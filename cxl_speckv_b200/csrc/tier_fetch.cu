// tier_fetch.cu -- kernels of the device-side tier fetch (speckv_ext_tier_fetch, tier.cu) and of the upkeep of the
// device copy of the tier's block directory.
//
// A fetch is lookup -> scan of the payload sizes -> gather over PCIe into HBM staging -> the codec's decoders on the
// staged (packed) container.  Nothing in it needs the host, so it can run inside a CUDA graph behind the prefetch
// kernels that produce the block ids.  Staging, rather than decoding straight out of host memory, keeps the tuned
// decoders as they are: they read their payload with TMA, and the generic second pass re-reads it.
#include <algorithm>

#include "device_ctx.h"
#include "tier_fetch.h"

namespace speckv {

namespace {

constexpr int kLookupThreads = 256;
constexpr int kGatherThreads = 256;
constexpr int kGatherVec = 8;                                               // 16-byte loads in flight per thread
constexpr uint64_t kGatherPiece = (uint64_t)kGatherThreads * kGatherVec * 16;   // 32 KiB of staging per CTA step
constexpr int kGatherCtasPerSm = 4;

// SET: request i names a block of a cache set; cache_index[i] >= n_caches is not served
template <bool SET>
__global__ void __launch_bounds__(kLookupThreads)
fetch_lookup_kernel(const DeviceDir* __restrict__ dir, const uint64_t* __restrict__ ids, const uint32_t* __restrict__ n_dev,
                    uint32_t n, uint32_t group_elems, int dtype, bool rle, uint64_t max_comp_bytes,
                    uint64_t* __restrict__ src_off, uint32_t* __restrict__ comp_bytes, float* __restrict__ scales,
                    uint8_t* __restrict__ status, const uint32_t* __restrict__ cache_index, uint32_t n_caches) {
    const uint32_t i = blockIdx.x * kLookupThreads + threadIdx.x;
    const uint32_t count = n_dev ? min(*n_dev, n) : n;
    if (i >= count) return;
    const DeviceDir d = *dir;
    const uint64_t key = ids[i];
    uint64_t off = 0;
    uint32_t cb = 0;
    float s = 1.0f;
    bool served = false;
    const bool in_set = !SET || cache_index[i] < n_caches;
    // the host map keeps its load under 0.7, so an empty slot ends every probe run; the bound only guards the loop
    for (uint64_t h = dir_hash(key) & d.mask, probes = 0; in_set && probes <= d.mask; h = (h + 1) & d.mask, ++probes) {
        const uint4* e = reinterpret_cast<const uint4*>(d.table + h);
        const uint4 lo = e[0];   // key, pool_off
        const uint4 hi = e[1];   // comp_bytes, scale, group_elems, dtype | scheme << 8 | ragged
        if ((int)hi.w == kDirEmpty) break;
        if (((uint64_t)lo.y << 32 | lo.x) != key) continue;
        const int rec = (int)hi.w, scheme = (rec >> 8) & 0xff;
        served = hi.z == group_elems && (rec & 0xff) == dtype && scheme != 0 && (scheme == 2 || scheme == 3) == rle &&
                 hi.x <= max_comp_bytes;
        if (served) {
            off = (uint64_t)lo.w << 32 | lo.z;
            cb = hi.x;
            s = __uint_as_float(hi.y);
        }
        break;
    }
    // an unserved request gets an empty payload: the decoders write nothing for it and report 0 elements
    src_off[i] = off;
    comp_bytes[i] = cb;
    scales[i] = s;
    if (status) status[i] = served ? 1 : 0;
}

// largest r in [lo, hi] with offsets[r] <= o (offsets ascending, offsets[lo] <= o).  Requests with an empty payload
// share their offset with the next one; the search lands on the last of them, the one whose bytes start there.
__device__ __forceinline__ uint32_t request_at(const uint64_t* __restrict__ offsets, uint32_t lo, uint32_t hi, uint64_t o) {
    while (lo < hi) {
        const uint32_t mid = lo + (hi - lo + 1) / 2;
        if (offsets[mid] <= o) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// Copies the staging range [0, *total) out of the pinned pool, balanced by bytes: a persistent grid walks the range in
// 32 KiB pieces (the total is known only on the device), every thread keeps kGatherVec 16-byte loads in flight to cover
// the microseconds of a PCIe read.  One search per piece finds the requests it spans; a piece inside one payload (blocks
// of 128 KiB and more) needs no per-load search.
__global__ void __launch_bounds__(kGatherThreads)
fetch_gather_kernel(const DeviceDir* __restrict__ dir, const uint64_t* __restrict__ src_off,
                    const uint64_t* __restrict__ offsets, const uint32_t* __restrict__ n_dev, uint32_t n,
                    const uint64_t* __restrict__ total_p, uint8_t* __restrict__ staging) {
    __shared__ uint32_t span[2];
    const uint32_t count = n_dev ? min(*n_dev, n) : n;
    const uint64_t total = *total_p;
    if (count == 0) return;
    const uint8_t* pool = dir->pool;
    for (uint64_t p0 = (uint64_t)blockIdx.x * kGatherPiece; p0 < total; p0 += (uint64_t)gridDim.x * kGatherPiece) {
        const uint64_t p1 = min(p0 + kGatherPiece, total);
        if (threadIdx.x == 0) {
            span[0] = request_at(offsets, 0, count - 1, p0);
            span[1] = request_at(offsets, span[0], count - 1, p1 - 1);
        }
        __syncthreads();
        const uint32_t r0 = span[0], r1 = span[1];
        __syncthreads();   // span is rewritten by the next piece
        uint4 v[kGatherVec];
#pragma unroll
        for (int u = 0; u < kGatherVec; ++u) {
            const uint64_t o = p0 + ((uint64_t)u * kGatherThreads + threadIdx.x) * 16;
            if (o < p1) {
                const uint32_t r = r0 == r1 ? r0 : request_at(offsets, r0, r1, o);
                v[u] = __ldg(reinterpret_cast<const uint4*>(pool + src_off[r] + (o - offsets[r])));
            }
        }
#pragma unroll
        for (int u = 0; u < kGatherVec; ++u) {
            const uint64_t o = p0 + ((uint64_t)u * kGatherThreads + threadIdx.x) * 16;
            if (o < p1) *reinterpret_cast<uint4*>(staging + o) = v[u];
        }
    }
}

__global__ void __launch_bounds__(256)
dir_apply_kernel(const DeviceDir* __restrict__ dir, const DirUpdate* __restrict__ upd, size_t n) {
    DirEntry* table = const_cast<DirEntry*>(dir->table);
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) table[upd[i].slot] = upd[i].e;
}

}  // namespace

cudaError_t launch_dir_apply(const DeviceDir* d_dir, const DirUpdate* d_upd, size_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const size_t grid = std::min<size_t>((n + 255) / 256, (size_t)current_sm_count() * 8);
    dir_apply_kernel<<<(unsigned)grid, 256, 0, st>>>(d_dir, d_upd, n);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_fetch_lookup(const DeviceDir* d_dir, const uint64_t* ids, const uint32_t* n_dev, uint32_t n,
                                uint32_t group_elems, int dtype, int scheme, size_t max_comp_bytes, uint64_t* src_off,
                                uint32_t* comp_bytes, float* scales, uint8_t* status, cudaStream_t st,
                                const uint32_t* cache_index, uint32_t n_caches) {
    const bool rle = scheme == 2 || scheme == 3;
    const unsigned grid = (n + kLookupThreads - 1) / kLookupThreads;
    if (cache_index)
        fetch_lookup_kernel<true><<<grid, kLookupThreads, 0, st>>>(d_dir, ids, n_dev, n, group_elems, dtype, rle, max_comp_bytes,
                                                                    src_off, comp_bytes, scales, status, cache_index, n_caches);
    else
        fetch_lookup_kernel<false><<<grid, kLookupThreads, 0, st>>>(d_dir, ids, n_dev, n, group_elems, dtype, rle, max_comp_bytes,
                                                                     src_off, comp_bytes, scales, status, nullptr, 0u);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_fetch_gather(const DeviceDir* d_dir, const uint64_t* src_off, const uint64_t* offsets,
                                const uint32_t* n_dev, uint32_t n, const uint64_t* total, uint8_t* staging,
                                int sm_count, cudaStream_t st) {
    fetch_gather_kernel<<<sm_count * kGatherCtasPerSm, kGatherThreads, 0, st>>>(d_dir, src_off, offsets, n_dev, n, total,
                                                                               staging);
    count_launch();
    return cudaGetLastError();
}

}  // namespace speckv
