// kv_codec_dispatch.cu -- picks the kernel family for a codec call.
//
// fp16/bf16 groups of R * 2048 elements (R a power of two up to 128) go to the tuned
// TMA/cluster kernels; every group those flag (runs of 8+ equal deltas, non-finite or
// tiny scales) and every other geometry goes to the generic kernel.  Both launches are
// ordered on the caller's stream; the flag array is a per-stream buffer the library keeps across calls.
#include <cstdlib>

#include "device_ctx.h"
#include "kv_codec.h"

namespace speckv {

static bool force_generic() {
    static const bool v = [] {
        const char* e = std::getenv("SPECKV_FORCE_GENERIC");
        return e && e[0] == '1';
    }();
    return v;
}

bool compress_packed_supported(const CodecArgs& a) {
    return !force_generic() && !a.group_len && scheme_is_rle(a.scheme) && fast_regions(a, false) == 1;
}

cudaError_t launch_compress(const CodecArgs& a, cudaStream_t st) {
    const int R = force_generic() ? 0 : fast_regions(a, false);
    if (a.pack_offsets) {
        // packed emission: one status word per CTA of the tuned kernel (16 page groups each), cleared for every launch
        if (!a.pack_total || !compress_packed_supported(a)) return cudaErrorInvalidValue;
        uint32_t* flags = nullptr;
        unsigned long long* status = nullptr;
        const size_t n_ctas = ((size_t)a.n_groups + 15) / 16;
        cudaError_t e = scratch_persistent(reinterpret_cast<void**>(&flags), (size_t)a.n_groups * sizeof(uint32_t), st);
        if (e == cudaSuccess) e = scratch_persistent(reinterpret_cast<void**>(&status), n_ctas * sizeof(unsigned long long), st, 2);
        if (e == cudaSuccess) e = cudaMemsetAsync(status, 0, n_ctas * sizeof(unsigned long long), st);
        if (e == cudaSuccess) e = launch_compress_fast(R, a, flags, st, status);
        CodecArgs second = a;
        second.slot_offsets = a.pack_offsets;   // the generic kernel writes into the whole slot reserved at pack_offsets[g]
        if (e == cudaSuccess) e = launch_compress_generic(second, st, flags);
        return e;
    }
    if (R == 0) return launch_compress_generic(a, st, nullptr);
    // the per-group flag words live in a buffer that belongs to the stream and stays allocated: no allocation on
    // the call path, and the two launches can be captured into a CUDA graph
    uint32_t* flags = nullptr;
    cudaError_t e = scratch_persistent(reinterpret_cast<void**>(&flags), (size_t)a.n_groups * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    e = launch_compress_fast(R, a, flags, st);
    if (e == cudaSuccess) e = launch_compress_generic(a, st, flags);
    return e;
}

cudaError_t launch_decompress(const CodecArgs& a, cudaStream_t st) {
    const int R = force_generic() ? 0 : fast_regions(a, true);
    if (R == 0) return launch_decompress_generic(a, st, nullptr, nullptr);
    // [counters 64 B][flags n][list n][prefix n * (R + 1)]: its own buffer (tag 1) -- the counters must stay zero
    // between calls, so nothing else may scribble here
    const size_t n = a.n_groups;
    const size_t off_flags = 64, off_list = off_flags + ((n * 4 + 15) & ~(size_t)15), off_prefix = off_list + ((n * 4 + 15) & ~(size_t)15);
    const bool rle = scheme_is_rle(a.scheme);
    const size_t bytes = off_prefix + (rle ? n * (size_t)(R + 1) * sizeof(uint2) : 0);
    uint8_t* base = nullptr;
    cudaError_t e = scratch_persistent(reinterpret_cast<void**>(&base), bytes, st, 1);
    if (e != cudaSuccess) return e;
    DecodeScratch sc;
    sc.counters = reinterpret_cast<uint32_t*>(base);
    sc.flags = reinterpret_cast<uint32_t*>(base + off_flags);
    sc.list = reinterpret_cast<uint32_t*>(base + off_list);
    sc.prefix = reinterpret_cast<uint2*>(base + off_prefix);
    sc.regions = (uint32_t)R;
    e = launch_decompress_fast(R, a, sc, st);
    if (e == cudaSuccess) e = launch_decompress_generic(a, st, sc.flags, rle ? &sc : nullptr);
    return e;
}

}  // namespace speckv
