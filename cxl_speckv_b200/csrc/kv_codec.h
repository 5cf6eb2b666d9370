// kv_codec.h -- internal launch interface between the C ABI (ext_api.cu) and the codec kernels.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace speckv {

// One codec call.  The host fills it and every codec kernel takes it by value: the container addressing below is
// written once, here, for all of them.
struct CodecArgs {
    const void* in = nullptr;        // compress: elements in; decompress: unused
    void* out = nullptr;             // decompress: elements out
    void* payload = nullptr;         // slots (written by compress, read by decompress)
    float* scales = nullptr;
    uint32_t* comp_bytes = nullptr;
    uint32_t* out_elems = nullptr;   // decompress, optional
    const uint32_t* src_index = nullptr;  // decompress, optional: output group i decodes payload group src_index[i]
    const uint64_t* slot_offsets = nullptr;  // optional: block b starts at payload + slot_offsets[b] (16 B aligned, packed
                                             // container) instead of b * slot_bytes.  Decompress, and the generic compress
                                             // behind a packed emission (the slots reserved at pack_offsets)
    const uint32_t* elem_index = nullptr;    // optional paged gather / scatter: group i's elements are block
                                             // elem_index[i] of the element buffer (compress reads `in` there,
                                             // decompress writes `out` there) instead of block i
    const uint32_t* n_groups_dev = nullptr;  // decompress, optional: device word holding the number of valid requests
                                             // (<= n_groups, which then is the capacity the grid is sized for)
    // compress, optional -- packed emission: the payloads go back to back (16 B aligned) into `payload` instead of
    // one slot per group; pack_offsets[g] receives the byte offset of group g, *pack_total the length of the stream.
    // Offsets follow from a look-back over per-CTA status words inside the compress kernel (no pack pass); a group
    // left to the generic kernel keeps a whole slot (its size is not known in the first pass).  Covered geometries:
    // compress_packed_supported().
    uint64_t* pack_offsets = nullptr;
    uint64_t* pack_total = nullptr;          // receives the stream length, or ~0 when the placement failed (look-back timeout)
    // compress, optional (device): group g encodes only the first min(group_len[g], group_elems) elements of its
    // block (the filled prefix of a paged KV block); no packed emission with it
    const uint32_t* group_len = nullptr;
    // optional KV cache set (speckv_ext_cache_set_create): group g's elements are block elem_index[g] of cache
    // cache_index[g], at cache_bases[cache_index[g]] + elem_index[g] * block_stride; `in` / `out` are unused.  Always
    // with elem_index.  An index >= n_caches addresses cache 0 (never read or written: the fetch leaves such a request
    // with an empty payload, and the other forms take it as a caller error)
    const uint64_t* cache_bases = nullptr;   // device: element address of each cache
    const uint32_t* cache_index = nullptr;   // device: per group
    uint64_t block_stride = 0;               // elements between consecutive blocks of a cache
    uint32_t n_caches = 0;
    bool set_unaligned = false;              // host: a base or the stride in bytes is not a multiple of 16 (generic kernels)
    size_t slot_bytes = 0;
    uint32_t group_elems = 0;
    uint32_t n_groups = 0;
    int dtype = 0;                   // DT_F16 / DT_BF16 / DT_F32
    int scheme = 2;                  // speckv_comp_scheme_t, or one of the extension ids 3 / 4 (speckv_ext.h)

    CodecArgs() = default;
    CodecArgs(size_t slot_bytes_, size_t group_elems_, size_t n_groups_, int dtype_, int scheme_)
        : slot_bytes(slot_bytes_), group_elems((uint32_t)group_elems_), n_groups((uint32_t)n_groups_), dtype(dtype_),
          scheme(scheme_) {}

    // ---- container addressing (device).  The index arrays stay unchanged during a launch: non-coherent loads.
    // group g's elements: block elem_index[g] of `base`, else block g (blocks of G elements); with a cache set, block
    // elem_index[g] of cache cache_index[g].  SET = false: a kernel instantiated for calls without a set (the generic
    // kernels have one instantiation per form, so that the set branch costs their single-cache forms nothing)
    template <bool SET = true, typename T>
    __device__ __forceinline__ T* elem_block(T* base, uint32_t g, uint32_t G) const {
        if (SET && cache_bases) {
            const uint32_t c = __ldg(cache_index + g);
            return reinterpret_cast<T*>(__ldg(cache_bases + (c < n_caches ? c : 0u))) +
                   (size_t)__ldg(elem_index + g) * block_stride;
        }
        return base + (size_t)(elem_index ? __ldg(elem_index + g) : g) * G;
    }
    // the stored block output group g decodes
    __device__ __forceinline__ uint32_t stored_block(uint32_t g) const { return src_index ? __ldg(src_index + g) : g; }
    // the payload of stored block b
    __device__ __forceinline__ uint8_t* block_payload(uint32_t b) const {
        return static_cast<uint8_t*>(payload) + (slot_offsets ? (size_t)__ldg(slot_offsets + b) : (size_t)b * slot_bytes);
    }
    // groups to process: n_groups, or fewer when the request count lives on the device
    __device__ __forceinline__ uint32_t live_groups() const { return n_groups_dev ? min(n_groups, __ldg(n_groups_dev)) : n_groups; }
    // elements group g encodes (blocks of G elements): a ragged call's filled prefix, else the whole block
    __device__ __forceinline__ uint32_t group_length(uint32_t g, uint32_t G) const {
        return group_len ? min(__ldg(group_len + g), G) : G;
    }
};

// scheme ids: 0 raw 16-bit passthrough, 1 codes only, 2 codes + delta + RLE (the reference's three), and the clamped
// variants of 2 and 1 that store s = max|x| (3, 4)
__host__ __device__ inline bool scheme_is_rle(int s) { return s == 2 || s == 3; }
__host__ __device__ inline bool scheme_is_codes(int s) { return s == 1 || s == 4; }
__host__ __device__ inline bool scheme_max_scale(int s) { return s == 3 || s == 4; }

// What the tuned decompress kernel leaves for the second pass (one buffer per stream, kept across calls):
//   flags[g]   0 = done, 1 = the generic kernel decodes group g, 2 = the run-expansion path does
//   list / counters[0]: the groups flagged 2, appended in any order; counters[1]: CTAs of the second pass that have
//              finished (the last one clears both, so the next call starts from zero without a memset)
//   prefix[g * (R + 1) + r] = (elements, code) before pairs-region r of group g; entry R = (decoded length, -)
struct DecodeScratch {
    uint32_t* flags = nullptr;
    uint32_t* list = nullptr;
    uint32_t* counters = nullptr;
    uint2* prefix = nullptr;
    uint32_t regions = 0;   // R of the call
};

// any geometry, any alignment (kv_codec_generic.cu)
// `only_flagged` (optional, device): process group g only if only_flagged[g] == 1
cudaError_t launch_compress_generic(const CodecArgs& a, cudaStream_t st, const uint32_t* only_flagged = nullptr);
cudaError_t launch_decompress_generic(const CodecArgs& a, cudaStream_t st, const uint32_t* only_flagged = nullptr,
                                      const DecodeScratch* runs = nullptr);

// tuned fp16/bf16 kernels for groups of R * 2048 elements (kv_codec_fast.cu).  fast_regions()
// returns R when they cover the call, else 0; they set flags[g] = 1 for every group they leave
// to the generic kernel.
int fast_regions(const CodecArgs& a, bool decompress);
bool compress_packed_supported(const CodecArgs& a);   // packed emission: fp16 / bf16 groups of 2048 elements (4 KiB pages), RLE schemes
struct PackOut {                                      // kernel-side view of the packed emission (all null = one slot per group)
    uint64_t* offsets = nullptr;
    uint64_t* total = nullptr;
    unsigned long long* status = nullptr;             // one word per CTA, zero before the launch
};
cudaError_t launch_compress_fast(int R, const CodecArgs& a, uint32_t* flags, cudaStream_t st, unsigned long long* pack_status = nullptr);
cudaError_t launch_decompress_fast(int R, const CodecArgs& a, const DecodeScratch& scratch, cudaStream_t st);

// dispatch: tuned kernels for the common geometries, generic otherwise (kv_codec_dispatch.cu)
cudaError_t launch_compress(const CodecArgs& a, cudaStream_t st);
cudaError_t launch_decompress(const CodecArgs& a, cudaStream_t st);

}  // namespace speckv
