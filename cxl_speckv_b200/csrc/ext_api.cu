// ext_api.cu -- the additive C ABI of libcxlspeckv.so (include/speckv_ext.h).
//
// Thin argument checking + dispatch onto the sm_100a kernels.  No torch types,
// no C++ types across the boundary.  There is no CPU fallback: without a usable
// CUDA device every entry point returns SPECKV_ERR_DRIVER.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/speckv_ext.h"
#include "atu.h"
#include "codec_math.cuh"
#include "device_ctx.h"
#include "kv_codec.h"

namespace speckv {

// ---- device context ---------------------------------------------------------------
static std::once_flag g_dev_once;
static int g_dev_count = 0;
static std::vector<int> g_sm_count;

static void probe_devices() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    g_dev_count = n;
    g_sm_count.assign(n > 0 ? n : 0, 148);
    for (int d = 0; d < n; ++d) {
        int sm = 0;
        if (cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, d) == cudaSuccess && sm > 0) g_sm_count[d] = sm;
    }
}

int device_count() {
    std::call_once(g_dev_once, probe_devices);
    return g_dev_count;
}

// Scratch for the codec calls (per-launch flag words) comes from a private stream-ordered pool that
// keeps its memory across synchronisations: the default pool releases everything at every sync, and
// the next cudaMallocAsync then pays a fresh physical allocation (measured: ~1 ms per first call).
static std::mutex g_pool_mu;
static std::vector<cudaMemPool_t> g_pools;

cudaError_t scratch_alloc(void** p, size_t bytes, cudaStream_t st) {
    if (device_count() <= 0) return cudaErrorNoDevice;
    int d = 0;
    cudaError_t e = cudaGetDevice(&d);
    if (e != cudaSuccess) return e;
    if (d < 0 || d >= g_dev_count) return cudaErrorInvalidDevice;
    cudaMemPool_t pool = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        if (g_pools.empty()) g_pools.assign(g_dev_count, nullptr);
        if (!g_pools[d]) {
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = d;
            e = cudaMemPoolCreate(&g_pools[d], &props);
            if (e != cudaSuccess) {
                g_pools[d] = nullptr;
                return e;
            }
            uint64_t keep = ~0ull;
            cudaMemPoolSetAttribute(g_pools[d], cudaMemPoolAttrReleaseThreshold, &keep);
        }
        pool = g_pools[d];
    }
    return cudaMallocFromPoolAsync(p, bytes, pool, st);
}

int current_sm_count() {
    if (device_count() <= 0) return 0;
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= g_dev_count) return 148;
    return g_sm_count[d];
}

speckv_status_t status_of(cudaError_t e) {
    if (e == cudaSuccess) return SPECKV_OK;
    cudaGetLastError();
    if (e == cudaErrorMemoryAllocation) return SPECKV_ERR_NOMEM;
    if (e == cudaErrorInvalidValue) return SPECKV_ERR_INVAL;
    return SPECKV_ERR_DRIVER;
}

// ---- statistics ---------------------------------------------------------------------
static std::atomic<uint64_t> g_n_comp{0}, g_n_decomp{0}, g_n_xlate{0}, g_b_comp{0}, g_b_decomp{0};
static std::atomic<uint64_t> g_b_h2d{0}, g_b_d2h{0};   // bytes the *_host calls moved over PCIe
std::atomic<uint64_t> g_kernel_launches{0};
void count_launch(unsigned n) { g_kernel_launches += n; }

static size_t elem_bytes(int dtype) { return dtype == DT_F32 ? 4 : 2; }

// Per-stream scratch that stays allocated across calls (the codec's per-group flag words): a call inside a
// serving loop then issues no allocation at all, and the launches can be captured into a CUDA graph.  The
// buffer of a (device, stream) pair only grows; growing is a plain cudaMalloc, which is refused while the
// stream is being captured -- run the call once before capturing it.
struct ScratchEntry {
    int device;
    int tag;
    cudaStream_t stream;
    void* ptr;
    size_t cap;
};
static std::mutex g_scratch_mu;
static std::vector<ScratchEntry> g_scratch;

cudaError_t scratch_persistent(void** p, size_t bytes, cudaStream_t st, int tag) {
    if (device_count() <= 0) return cudaErrorNoDevice;
    int d = 0;
    cudaError_t e = cudaGetDevice(&d);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    ScratchEntry* hit = nullptr;
    for (ScratchEntry& s : g_scratch)
        if (s.device == d && s.stream == st && s.tag == tag) hit = &s;
    if (hit && hit->cap >= bytes) {
        *p = hit->ptr;
        return cudaSuccess;
    }
    size_t cap = 4096;
    while (cap < bytes) cap *= 2;
    void* np = nullptr;
    if ((e = cudaMalloc(&np, cap)) != cudaSuccess) return e;
    if ((e = cudaMemset(np, 0, cap)) != cudaSuccess) {   // counters kept in such buffers start at zero
        cudaFree(np);
        return e;
    }
    if (hit) {
        cudaFree(hit->ptr);   // synchronises: earlier launches on the stream that use the old buffer have finished
        hit->ptr = np;
        hit->cap = cap;
    } else {
        if (g_scratch.size() >= 256) {   // streams come and go: recycle the oldest entry
            cudaFree(g_scratch.front().ptr);
            g_scratch.erase(g_scratch.begin());
        }
        g_scratch.push_back(ScratchEntry{d, tag, st, np, cap});
    }
    *p = np;
    return cudaSuccess;
}

// ---- engine latency statistics (EngineStatistics::avg_*_latency_ns, cache_engine.cpp:65-79,103-112) ----
// The reference brackets every compress() / decompress() call with a steady_clock pair and keeps a running mean.
// The calls here are asynchronous, so the bracket is a pair of CUDA events on the caller's stream; finished
// pairs are harvested lazily (no synchronisation on the call path).  Calls made while the stream is being
// captured into a graph are not timed (events recorded in a capture cannot be queried).
struct LatencyPair {
    cudaEvent_t a = nullptr, b = nullptr;
    int device = -1;
    bool decompress = false, busy = false;
    uint64_t groups = 0, bytes = 0;
};
static std::mutex g_lat_mu;
static LatencyPair g_lat[64];
static double g_lat_ns[2] = {0.0, 0.0}, g_lat_mean_ns[2] = {0.0, 0.0};   // [0] compress, [1] decompress
static uint64_t g_lat_calls[2] = {0, 0}, g_lat_groups[2] = {0, 0}, g_lat_bytes[2] = {0, 0};
static double g_ratio_mean = 0.0;      // running mean of original_size / compressed_size over groups
static uint64_t g_ratio_groups = 0;
static const bool g_lat_enabled = [] {
    const char* e = std::getenv("SPECKV_LATENCY_STATS");
    return !(e && e[0] == '0');
}();

static void latency_harvest_locked(bool wait) {
    for (LatencyPair& p : g_lat) {
        if (!p.busy) continue;
        cudaError_t q = wait ? cudaEventSynchronize(p.b) : cudaEventQuery(p.b);
        if (q == cudaErrorNotReady) continue;
        float ms = 0.0f;
        if (q == cudaSuccess && cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            const int k = p.decompress ? 1 : 0;
            g_lat_ns[k] += (double)ms * 1e6;
            ++g_lat_calls[k];
            g_lat_groups[k] += p.groups;
            g_lat_bytes[k] += p.bytes;
            // the reference's update rule, one step per call (cache_engine.cpp:76-79)
            g_lat_mean_ns[k] = (g_lat_mean_ns[k] * (double)(g_lat_calls[k] - 1) + (double)ms * 1e6) / (double)g_lat_calls[k];
        } else {
            cudaGetLastError();
        }
        p.busy = false;
    }
}

class LatencyScope {
public:
    LatencyScope(bool decompress, cudaStream_t st, uint64_t groups = 0, uint64_t bytes = 0) : st_(st) {
        if (!g_lat_enabled) return;
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
            cudaGetLastError();
            return;
        }
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return;
        std::lock_guard<std::mutex> lk(g_lat_mu);
        for (int pass = 0; pass < 2 && !p_; ++pass) {
            for (LatencyPair& p : g_lat)
                if (!p.busy && (p.device == dev || p.device < 0)) {
                    p_ = &p;
                    break;
                }
            if (!p_) latency_harvest_locked(false);
        }
        if (!p_) return;   // every pair still in flight: this call goes untimed
        if (!p_->a) {
            if (cudaEventCreate(&p_->a) != cudaSuccess || cudaEventCreate(&p_->b) != cudaSuccess) {
                cudaGetLastError();
                p_ = nullptr;
                return;
            }
            p_->device = dev;
        }
        p_->busy = true;
        p_->decompress = decompress;
        p_->groups = groups;
        p_->bytes = bytes;
        cudaEventRecord(p_->a, st_);
    }
    ~LatencyScope() {
        if (p_) cudaEventRecord(p_->b, st_);
    }
    void set_groups(uint64_t g) {
        if (p_) p_->groups = g;
    }

private:
    cudaStream_t st_;
    LatencyPair* p_ = nullptr;
};

static bool valid_common(int dtype, size_t group_elems, size_t n_groups, size_t slot_bytes, int scheme) {
    if (dtype < 0 || dtype > 2 || scheme < 0 || scheme > 4) return false;
    if (group_elems >= (1ull << 31) || n_groups >= (1ull << 32)) return false;
    if (scheme == 0 && dtype == DT_F32) return false;  // FP16 scheme is a raw 16-bit passthrough
    if (slot_bytes % 16 != 0 || slot_bytes < speckv_ext_slot_bytes(group_elems, (speckv_comp_scheme_t)scheme)) return false;
    if (slot_bytes >= (1ull << 32)) return false;
    return true;
}

// ---- pipelined host-buffer path --------------------------------------------------------
struct HostPipe {
    static constexpr int kSlots = 3;
    std::mutex mu;
    int device = -1;
    cudaStream_t st[kSlots] = {};
    cudaEvent_t ev_meta[kSlots] = {};   // "the sizes of this slot's chunk are on the host"
    void* d_elems[kSlots] = {};
    void* d_payload[kSlots] = {};
    float* d_scales[kSlots] = {};
    uint32_t* d_comp[kSlots] = {};
    uint32_t* d_oel[kSlots] = {};
    size_t cap_elems = 0, cap_payload = 0, cap_groups = 0;

    void release() {
        for (int i = 0; i < kSlots; ++i) {
            if (d_elems[i]) cudaFree(d_elems[i]);
            if (d_payload[i]) cudaFree(d_payload[i]);
            if (d_scales[i]) cudaFree(d_scales[i]);
            if (d_comp[i]) cudaFree(d_comp[i]);
            if (d_oel[i]) cudaFree(d_oel[i]);
            d_elems[i] = d_payload[i] = nullptr;
            d_scales[i] = nullptr;
            d_comp[i] = d_oel[i] = nullptr;
        }
        cap_elems = cap_payload = cap_groups = 0;
    }

    cudaError_t ensure(size_t elems_bytes, size_t payload_bytes, size_t groups) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        if (dev != device) {
            release();
            for (int i = 0; i < kSlots; ++i) {
                if (st[i]) cudaStreamDestroy(st[i]);
                if (ev_meta[i]) cudaEventDestroy(ev_meta[i]);
                st[i] = nullptr;
                ev_meta[i] = nullptr;
            }
            device = dev;
        }
        for (int i = 0; i < kSlots; ++i) {
            if (!st[i] && (e = cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking)) != cudaSuccess) return e;
            if (!ev_meta[i] && (e = cudaEventCreateWithFlags(&ev_meta[i], cudaEventDisableTiming)) != cudaSuccess) return e;
        }
        if (elems_bytes > cap_elems || payload_bytes > cap_payload || groups > cap_groups) {
            release();
            for (int i = 0; i < kSlots; ++i) {
                if ((e = cudaMalloc(&d_elems[i], elems_bytes)) != cudaSuccess) return e;
                if ((e = cudaMalloc(&d_payload[i], payload_bytes)) != cudaSuccess) return e;
                if ((e = cudaMalloc((void**)&d_scales[i], groups * sizeof(float))) != cudaSuccess) return e;
                if ((e = cudaMalloc((void**)&d_comp[i], groups * sizeof(uint32_t))) != cudaSuccess) return e;
                if ((e = cudaMalloc((void**)&d_oel[i], groups * sizeof(uint32_t))) != cudaSuccess) return e;
            }
            cap_elems = elems_bytes;
            cap_payload = payload_bytes;
            cap_groups = groups;
        }
        return cudaSuccess;
    }
};
static HostPipe g_pipe;

void release_host_pipe() {
    std::lock_guard<std::mutex> lk(g_pipe.mu);
    g_pipe.release();
}

// groups per chunk: aim at ~32 MiB of elements so H2D, kernel and D2H of neighbouring chunks overlap
static size_t chunk_groups(size_t group_bytes, size_t n_groups) {
    static const size_t target = [] {
        const char* e = std::getenv("SPECKV_HOST_CHUNK_MIB");
        const long v = e ? std::atol(e) : 0;
        return (size_t)(v > 0 ? v : 64) << 20;
    }();
    size_t c = group_bytes ? target / group_bytes : n_groups;
    if (c < 1) c = 1;
    if (c > n_groups) c = n_groups;
    return c ? c : 1;
}

// Payload copies of the host-buffer calls.  The slots of a chunk are mostly empty when the data compresses, so the
// copy follows the sizes: one copy of all slots when they are nearly full (or the groups are many and small: a
// driver call per group would cost more than the bytes it saves), else one copy per group of just its payload
// (rounded up to 16 bytes, never past the slot).  Returns the bytes moved.
static uint64_t copy_payloads(void* dst, const void* src, size_t slot_bytes, const uint32_t* h_comp, size_t ng,
                              cudaMemcpyKind kind, cudaStream_t st, cudaError_t& e) {
    uint64_t sum = 0;
    for (size_t g = 0; g < ng; ++g) sum += std::min<uint64_t>(((uint64_t)h_comp[g] + 15u) & ~15ull, slot_bytes);
    if (ng > 4096 || sum * 4 >= (uint64_t)ng * slot_bytes * 3) {
        e = cudaMemcpyAsync(dst, src, ng * slot_bytes, kind, st);
        return (uint64_t)ng * slot_bytes;
    }
    for (size_t g = 0; g < ng && e == cudaSuccess; ++g) {
        const size_t len = std::min<uint64_t>(((uint64_t)h_comp[g] + 15u) & ~15ull, slot_bytes);
        if (len) e = cudaMemcpyAsync((char*)dst + g * slot_bytes, (const char*)src + g * slot_bytes, len, kind, st);
    }
    return sum;
}

// sum of payload sizes and sum of the per-group ratios original_size / compressed_size, where
// original_size = n * sizeof(float) exactly as the reference accounts it (cache_engine.cpp:49,72)
__global__ void __launch_bounds__(256)
ratio_kernel(const uint32_t* __restrict__ comp_bytes, size_t n_groups, double original_bytes, double* __restrict__ acc) {
    double c = 0.0, r = 0.0;
    for (size_t g = (size_t)blockIdx.x * 256 + threadIdx.x; g < n_groups; g += (size_t)gridDim.x * 256) {
        const double cb = (double)comp_bytes[g];
        c += cb;
        if (cb > 0.0) r += original_bytes / cb;
    }
    for (int o = 16; o > 0; o >>= 1) {
        c += __shfl_xor_sync(0xffffffffu, c, o);
        r += __shfl_xor_sync(0xffffffffu, r, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&acc[0], c);
        atomicAdd(&acc[1], r);
    }
}

}  // namespace speckv

using namespace speckv;

extern "C" {

speckv_status_t speckv_ext_ratio_stats(const uint32_t* d_comp_bytes, size_t n_groups, size_t group_elems,
                                       double* out_total_comp_bytes, double* out_mean_ratio, void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!d_comp_bytes || !out_total_comp_bytes || !out_mean_ratio) return SPECKV_ERR_INVAL;
    *out_total_comp_bytes = 0.0;
    *out_mean_ratio = 0.0;
    if (n_groups == 0) return SPECKV_OK;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    double* d_acc = nullptr;
    cudaError_t e = scratch_alloc((void**)&d_acc, 16, st);
    if (e != cudaSuccess) return status_of(e);
    cudaMemsetAsync(d_acc, 0, 16, st);
    size_t blocks = (n_groups + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    ratio_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_comp_bytes, n_groups, (double)group_elems * 4.0, d_acc);
    count_launch();
    double h[2] = {0.0, 0.0};
    e = cudaMemcpyAsync(h, d_acc, 16, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFreeAsync(d_acc, st);
    *out_total_comp_bytes = h[0];
    *out_mean_ratio = h[1] / (double)n_groups;
    if (e == cudaSuccess) {   // EngineStatistics::avg_compression_ratio: running mean over every group reported here
        std::lock_guard<std::mutex> lk(g_lat_mu);
        g_ratio_mean = (g_ratio_mean * (double)g_ratio_groups + h[1]) / (double)(g_ratio_groups + n_groups);
        g_ratio_groups += n_groups;
    }
    return status_of(e);
}

int speckv_ext_device_count(void) { return device_count(); }

const char* speckv_ext_version(void) { return "cxl-speckv-b200 0.1 (sm_100a)"; }

size_t speckv_ext_slot_bytes(size_t group_elems, speckv_comp_scheme_t scheme) {
    size_t b = ((int)scheme == SPECKV_COMP_INT8 || (int)scheme == SPECKV_COMP_INT8_CLAMP) ? group_elems : 2 * group_elems;
    return (b + 15) / 16 * 16;
}

// ---- device-buffer codec entry points: one marshalling routine for all of them ----------------------
}  // extern "C"

namespace speckv {
// validation shared by every codec call + the fields every call fills the same way
static speckv_status_t codec_args(CodecArgs& a, int dtype, size_t group_elems, size_t n_groups, const void* d_payload,
                                  size_t slot_bytes, const float* d_scales, const uint32_t* d_comp_bytes, int scheme,
                                  const void* d_elems) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!valid_common(dtype, group_elems, n_groups, slot_bytes, scheme)) return SPECKV_ERR_INVAL;
    if (n_groups == 0) return SPECKV_OK;
    if (!d_payload || !d_scales || !d_comp_bytes || (!d_elems && group_elems)) return SPECKV_ERR_INVAL;
    if (reinterpret_cast<uintptr_t>(d_payload) & 15) return SPECKV_ERR_INVAL;
    a = CodecArgs(slot_bytes, group_elems, n_groups, dtype, scheme);
    a.payload = const_cast<void*>(d_payload);
    a.scales = const_cast<float*>(d_scales);
    a.comp_bytes = const_cast<uint32_t*>(d_comp_bytes);
    return SPECKV_OK;
}
static speckv_status_t codec_run(bool decompress, const CodecArgs& a, void* cuda_stream) {
    if (a.n_groups == 0) return SPECKV_OK;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    LatencyScope lat(decompress, st, a.n_groups, (uint64_t)a.n_groups * a.group_elems * elem_bytes(a.dtype));
    const cudaError_t e = decompress ? launch_decompress(a, st) : launch_compress(a, st);
    if (e == cudaSuccess) {
        (decompress ? g_n_decomp : g_n_comp) += a.n_groups;
        (decompress ? g_b_decomp : g_b_comp) += (uint64_t)a.n_groups * a.group_elems * elem_bytes(a.dtype);
    }
    return status_of(e);
}
}  // namespace speckv

extern "C" {

speckv_status_t speckv_ext_compress(const void* d_in, speckv_dtype_t dtype, size_t group_elems, size_t n_groups,
                                    void* d_payload, size_t slot_bytes, float* d_scales, uint32_t* d_comp_bytes,
                                    speckv_comp_scheme_t scheme, void* cuda_stream) {
    CodecArgs a;
    const speckv_status_t rc = codec_args(a, dtype, group_elems, n_groups, d_payload, slot_bytes, d_scales, d_comp_bytes, scheme, d_in);
    if (rc != SPECKV_OK) return rc;
    a.in = d_in;
    return codec_run(false, a, cuda_stream);
}

speckv_status_t speckv_ext_decompress(const void* d_payload, size_t slot_bytes, const float* d_scales,
                                      const uint32_t* d_comp_bytes, size_t group_elems, size_t n_groups,
                                      speckv_dtype_t dtype, void* d_out, uint32_t* d_out_elems,
                                      speckv_comp_scheme_t scheme, void* cuda_stream) {
    CodecArgs a;
    const speckv_status_t rc = codec_args(a, dtype, group_elems, n_groups, d_payload, slot_bytes, d_scales, d_comp_bytes, scheme, d_out);
    if (rc != SPECKV_OK) return rc;
    a.out = d_out;
    a.out_elems = d_out_elems;
    return codec_run(true, a, cuda_stream);
}

speckv_status_t speckv_ext_decompress_indexed(const void* d_payload, size_t slot_bytes, const float* d_scales,
                                              const uint32_t* d_comp_bytes, const uint32_t* d_block_index,
                                              size_t n_requests, size_t group_elems, speckv_dtype_t dtype, void* d_out,
                                              uint32_t* d_out_elems, speckv_comp_scheme_t scheme, void* cuda_stream) {
    CodecArgs a;
    const speckv_status_t rc = codec_args(a, dtype, group_elems, n_requests, d_payload, slot_bytes, d_scales, d_comp_bytes, scheme, d_out);
    if (rc != SPECKV_OK) return rc;
    if (n_requests && !d_block_index) return SPECKV_ERR_INVAL;
    a.out = d_out;
    a.out_elems = d_out_elems;
    a.src_index = d_block_index;
    return codec_run(true, a, cuda_stream);
}

speckv_status_t speckv_ext_decompress_routed(const void* d_payload, size_t slot_bytes, const float* d_scales,
                                             const uint32_t* d_comp_bytes, const uint32_t* d_block_index,
                                             const uint32_t* d_n_requests, size_t max_requests, size_t group_elems,
                                             speckv_dtype_t dtype, void* d_out, uint32_t* d_out_elems,
                                             speckv_comp_scheme_t scheme, void* cuda_stream) {
    CodecArgs a;
    const speckv_status_t rc = codec_args(a, dtype, group_elems, max_requests, d_payload, slot_bytes, d_scales, d_comp_bytes, scheme, d_out);
    if (rc != SPECKV_OK) return rc;
    if (max_requests && (!d_block_index || !d_n_requests)) return SPECKV_ERR_INVAL;
    a.out = d_out;
    a.out_elems = d_out_elems;
    a.src_index = d_block_index;
    a.n_groups_dev = d_n_requests;
    return codec_run(true, a, cuda_stream);
}

speckv_status_t speckv_ext_compress_gather(const void* d_cache, const uint32_t* d_block_table, speckv_dtype_t dtype,
                                           size_t group_elems, size_t n_groups, void* d_payload, size_t slot_bytes,
                                           float* d_scales, uint32_t* d_comp_bytes, speckv_comp_scheme_t scheme,
                                           void* cuda_stream) {
    if (scheme == SPECKV_COMP_FP16) return device_count() <= 0 ? SPECKV_ERR_DRIVER : SPECKV_ERR_INVAL;
    CodecArgs a;
    const speckv_status_t rc = codec_args(a, dtype, group_elems, n_groups, d_payload, slot_bytes, d_scales, d_comp_bytes, scheme, d_cache);
    if (rc != SPECKV_OK) return rc;
    if (n_groups && !d_block_table) return SPECKV_ERR_INVAL;
    a.in = d_cache;
    a.elem_index = d_block_table;
    return codec_run(false, a, cuda_stream);
}

speckv_status_t speckv_ext_compress_ragged(const void* d_in, const uint32_t* d_block_table, const uint32_t* d_group_len,
                                           speckv_dtype_t dtype, size_t group_elems, size_t n_groups, void* d_payload,
                                           size_t slot_bytes, float* d_scales, uint32_t* d_comp_bytes,
                                           speckv_comp_scheme_t scheme, void* cuda_stream) {
    if (scheme == SPECKV_COMP_FP16) return device_count() <= 0 ? SPECKV_ERR_DRIVER : SPECKV_ERR_INVAL;
    CodecArgs a;
    const speckv_status_t rc = codec_args(a, dtype, group_elems, n_groups, d_payload, slot_bytes, d_scales, d_comp_bytes, scheme, d_in);
    if (rc != SPECKV_OK) return rc;
    if (n_groups && !d_group_len) return SPECKV_ERR_INVAL;
    a.in = d_in;
    a.elem_index = d_block_table;
    a.group_len = d_group_len;
    return codec_run(false, a, cuda_stream);
}

speckv_status_t speckv_ext_decompress_scatter(const void* d_payload, size_t slot_bytes, const float* d_scales,
                                              const uint32_t* d_comp_bytes, const uint32_t* d_src_index,
                                              const uint32_t* d_block_table, size_t n_requests, size_t group_elems,
                                              speckv_dtype_t dtype, void* d_cache, uint32_t* d_out_elems,
                                              speckv_comp_scheme_t scheme, void* cuda_stream) {
    if (scheme == SPECKV_COMP_FP16) return device_count() <= 0 ? SPECKV_ERR_DRIVER : SPECKV_ERR_INVAL;
    CodecArgs a;
    const speckv_status_t rc = codec_args(a, dtype, group_elems, n_requests, d_payload, slot_bytes, d_scales, d_comp_bytes, scheme, d_cache);
    if (rc != SPECKV_OK) return rc;
    if (n_requests && !d_block_table) return SPECKV_ERR_INVAL;
    a.out = d_cache;
    a.elem_index = d_block_table;
    a.out_elems = d_out_elems;
    a.src_index = d_src_index;
    return codec_run(true, a, cuda_stream);
}

speckv_status_t speckv_ext_compress_host(const void* h_in, speckv_dtype_t dtype, size_t group_elems, size_t n_groups,
                                         void* h_payload, size_t slot_bytes, float* h_scales, uint32_t* h_comp_bytes,
                                         speckv_comp_scheme_t scheme) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!valid_common(dtype, group_elems, n_groups, slot_bytes, scheme)) return SPECKV_ERR_INVAL;
    if (n_groups == 0) return SPECKV_OK;
    if (!h_in || !h_payload || !h_scales || !h_comp_bytes) return SPECKV_ERR_INVAL;
    const size_t gbytes = group_elems * elem_bytes(dtype);
    const size_t cg = chunk_groups(gbytes > slot_bytes ? gbytes : slot_bytes, n_groups);
    std::lock_guard<std::mutex> lk(g_pipe.mu);
    cudaError_t e = g_pipe.ensure(cg * gbytes + 16, cg * slot_bytes, cg);
    if (e != cudaSuccess) return status_of(e);
    size_t chunk = 0;
    uint64_t moved_up = 0, moved_down = 0;
    // the payload copy of a chunk is issued one chunk later, once its sizes have reached the host: the copy then
    // moves the payload bytes, not the worst-case slots
    size_t prev_g0 = 0, prev_ng = 0;
    int prev_k = -1;
    auto finish = [&](size_t g0, size_t ng, int k) {
        cudaError_t e2 = cudaEventSynchronize(g_pipe.ev_meta[k]);
        if (e2 == cudaSuccess)
            moved_down += copy_payloads((char*)h_payload + g0 * slot_bytes, g_pipe.d_payload[k], slot_bytes, h_comp_bytes + g0, ng,
                                        cudaMemcpyDeviceToHost, g_pipe.st[k], e2);
        return e2;
    };
    for (size_t g0 = 0; g0 < n_groups; g0 += cg, ++chunk) {
        const size_t ng = (n_groups - g0 < cg) ? n_groups - g0 : cg;
        const int k = (int)(chunk % HostPipe::kSlots);
        cudaStream_t st = g_pipe.st[k];
        if ((e = cudaMemcpyAsync(g_pipe.d_elems[k], (const char*)h_in + g0 * gbytes, ng * gbytes, cudaMemcpyHostToDevice, st)) != cudaSuccess) break;
        moved_up += ng * gbytes;
        CodecArgs a(slot_bytes, group_elems, ng, dtype, scheme);
        a.in = g_pipe.d_elems[k];
        a.payload = g_pipe.d_payload[k];
        a.scales = g_pipe.d_scales[k];
        a.comp_bytes = g_pipe.d_comp[k];
        if ((e = launch_compress(a, st)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(h_comp_bytes + g0, g_pipe.d_comp[k], ng * sizeof(uint32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
        if ((e = cudaEventRecord(g_pipe.ev_meta[k], st)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(h_scales + g0, g_pipe.d_scales[k], ng * sizeof(float), cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
        moved_down += ng * 8;
        if (prev_k >= 0 && (e = finish(prev_g0, prev_ng, prev_k)) != cudaSuccess) break;
        prev_g0 = g0;
        prev_ng = ng;
        prev_k = k;
    }
    if (e == cudaSuccess && prev_k >= 0) e = finish(prev_g0, prev_ng, prev_k);
    for (int k = 0; k < HostPipe::kSlots; ++k) {
        cudaError_t e2 = cudaStreamSynchronize(g_pipe.st[k]);
        if (e == cudaSuccess) e = e2;
    }
    if (e == cudaSuccess) {
        g_n_comp += n_groups;
        g_b_comp += (uint64_t)n_groups * gbytes;
        g_b_h2d += moved_up;
        g_b_d2h += moved_down;
    }
    return status_of(e);
}

speckv_status_t speckv_ext_decompress_host(const void* h_payload, size_t slot_bytes, const float* h_scales,
                                           const uint32_t* h_comp_bytes, size_t group_elems, size_t n_groups,
                                           speckv_dtype_t dtype, void* h_out, uint32_t* h_out_elems,
                                           speckv_comp_scheme_t scheme) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!valid_common(dtype, group_elems, n_groups, slot_bytes, scheme)) return SPECKV_ERR_INVAL;
    if (n_groups == 0) return SPECKV_OK;
    if (!h_payload || !h_scales || !h_comp_bytes || !h_out) return SPECKV_ERR_INVAL;
    const size_t gbytes = group_elems * elem_bytes(dtype);
    const size_t cg = chunk_groups(gbytes > slot_bytes ? gbytes : slot_bytes, n_groups);
    std::lock_guard<std::mutex> lk(g_pipe.mu);
    cudaError_t e = g_pipe.ensure(cg * gbytes + 16, cg * slot_bytes, cg);
    if (e != cudaSuccess) return status_of(e);
    uint64_t moved_up = 0, moved_down = 0;
    size_t chunk = 0;
    for (size_t g0 = 0; g0 < n_groups; g0 += cg, ++chunk) {
        const size_t ng = (n_groups - g0 < cg) ? n_groups - g0 : cg;
        const int k = (int)(chunk % HostPipe::kSlots);
        cudaStream_t st = g_pipe.st[k];
        moved_up += copy_payloads(g_pipe.d_payload[k], (const char*)h_payload + g0 * slot_bytes, slot_bytes, h_comp_bytes + g0, ng,
                                  cudaMemcpyHostToDevice, st, e);
        if (e != cudaSuccess) break;
        moved_up += ng * 8;
        moved_down += ng * gbytes + (h_out_elems ? ng * 4 : 0);
        if ((e = cudaMemcpyAsync(g_pipe.d_scales[k], h_scales + g0, ng * sizeof(float), cudaMemcpyHostToDevice, st)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(g_pipe.d_comp[k], h_comp_bytes + g0, ng * sizeof(uint32_t), cudaMemcpyHostToDevice, st)) != cudaSuccess) break;
        CodecArgs a(slot_bytes, group_elems, ng, dtype, scheme);
        a.out = g_pipe.d_elems[k];
        a.payload = g_pipe.d_payload[k];
        a.scales = g_pipe.d_scales[k];
        a.comp_bytes = g_pipe.d_comp[k];
        a.out_elems = g_pipe.d_oel[k];
        if ((e = launch_decompress(a, st)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync((char*)h_out + g0 * gbytes, g_pipe.d_elems[k], ng * gbytes, cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
        if (h_out_elems && (e = cudaMemcpyAsync(h_out_elems + g0, g_pipe.d_oel[k], ng * sizeof(uint32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
    }
    for (int k = 0; k < HostPipe::kSlots; ++k) {
        cudaError_t e2 = cudaStreamSynchronize(g_pipe.st[k]);
        if (e == cudaSuccess) e = e2;
    }
    if (e == cudaSuccess) {
        g_n_decomp += n_groups;
        g_b_decomp += (uint64_t)n_groups * gbytes;
        g_b_h2d += moved_up;
        g_b_d2h += moved_down;
    }
    return status_of(e);
}

void* speckv_ext_host_alloc(size_t bytes) {
    if (device_count() <= 0) return nullptr;
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void speckv_ext_host_free(void* p) {
    if (p && device_count() > 0) cudaFreeHost(p);
}

speckv_status_t speckv_ext_translate(const uint64_t* d_va, uint64_t* d_pa, size_t n, void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (n == 0) return SPECKV_OK;
    if (!d_va || !d_pa) return SPECKV_ERR_INVAL;
    cudaError_t e = launch_translate(d_va, d_pa, n, current_sm_count(), static_cast<cudaStream_t>(cuda_stream));
    if (e == cudaSuccess) g_n_xlate += n;
    return status_of(e);
}

void speckv_ext_get_stats(speckv_ext_stats_t* out) {
    if (!out) return;
    out->total_compressions = g_n_comp.load();
    out->total_decompressions = g_n_decomp.load();
    out->total_translations = g_n_xlate.load();
    out->bytes_in_compress = g_b_comp.load();
    out->bytes_out_decompress = g_b_decomp.load();
    out->kernel_launches = g_kernel_launches.load();
    out->host_api_h2d_bytes = g_b_h2d.load();
    out->host_api_d2h_bytes = g_b_d2h.load();
}

void speckv_ext_engine_stats(speckv_engine_stats_t* out, int wait) {
    if (!out) return;
    std::memset(out, 0, sizeof(*out));
    std::lock_guard<std::mutex> lk(g_lat_mu);
    if (device_count() > 0) latency_harvest_locked(wait != 0);
    out->total_compressions = g_n_comp.load();
    out->total_decompressions = g_n_decomp.load();
    out->avg_compression_ratio = g_ratio_mean;
    out->avg_compression_latency_ns = g_lat_mean_ns[0];
    out->avg_decompression_latency_ns = g_lat_mean_ns[1];
    out->compress_calls_timed = g_lat_calls[0];
    out->decompress_calls_timed = g_lat_calls[1];
    out->compress_ns_per_group = g_lat_groups[0] ? g_lat_ns[0] / (double)g_lat_groups[0] : 0.0;
    out->decompress_ns_per_group = g_lat_groups[1] ? g_lat_ns[1] / (double)g_lat_groups[1] : 0.0;
    const double ns = g_lat_ns[0] + g_lat_ns[1];
    // the reference returns a constant here (512 bit x 800 MHz, cache_engine.cpp:291-296); this is measured:
    // uncompressed bytes through the timed calls per second of device time
    out->throughput_gbps = ns > 0.0 ? (double)(g_lat_bytes[0] + g_lat_bytes[1]) * 8.0 / ns : 0.0;
}

void speckv_ext_reset_stats(void) {
    {
        std::lock_guard<std::mutex> lk(g_lat_mu);
        if (device_count() > 0) latency_harvest_locked(false);
        for (int k = 0; k < 2; ++k) {
            g_lat_ns[k] = g_lat_mean_ns[k] = 0.0;
            g_lat_calls[k] = g_lat_groups[k] = g_lat_bytes[k] = 0;
        }
        g_ratio_mean = 0.0;
        g_ratio_groups = 0;
    }
    g_n_comp = 0;
    g_n_decomp = 0;
    g_n_xlate = 0;
    g_b_comp = 0;
    g_b_decomp = 0;
    g_b_h2d = 0;
    g_b_d2h = 0;
    g_kernel_launches = 0;
}

}  // extern "C"
