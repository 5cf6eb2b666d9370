// kv_codec_fast.cu -- KV block codec, tuned sm_100a path for fp16/bf16 groups of
// R * 2048 elements (R = 1, 2, 4 ... 128; the 4 KiB page group and the
// 1024-token x 128-dim block are R = 1 and R = 64).
//
// Geometry.  A *region* is 2048 consecutive elements (compress) or 2048
// consecutive [value][count] pairs (decompress): 4 KiB, owned by one warp and
// brought into shared memory by ONE bulk-TMA copy (cp.async.bulk, completion on
// a per-warp mbarrier).  A CTA has 16 warps = 16 regions = 64 KiB of tiles.
// A group of R regions is R warps of one CTA (R <= 16; 16/R groups per CTA) or a
// thread-block cluster of R/16 CTAs (R = 32/64/128 -> clusters of 2/4/8) whose
// CTAs exchange one word per region through distributed shared memory:
//   * the region max-abs  (group scale, cache_engine.cpp:172-184)
//   * the region run-head count / the region (sum count, sum value*count)
//     (exclusive sums give every region its output offset and, for decode, its
//     starting code), so delta + RLE still run over the whole flat group exactly
//     as the reference's sequential loops do (cache_engine.cpp:198-273).
// HBM traffic is the algorithmic minimum: each input byte is read once (TMA ->
// smem, max-abs and quantisation both read the smem tile), each output byte is
// written once: the staged region leaves shared memory with one bulk-TMA store.
//
// The common path is built for what holds for KV activations: no run of equal deltas
// spans a whole 8-element lane chunk (compress) / counts of 1 and 2 (decompress).
// Groups with longer runs take the long-run routines of this file (compress) or the
// run-expansion path of the second launch (decompress); zero groups are written in
// closed form.  What remains -- +-inf, tiny or huge bf16 scales, malformed payloads --
// is flagged in `needs_generic` and re-done by the generic kernel
// (kv_codec_generic.cu) in the same stream, so results are bit-exact for every input.
// Page groups (R = 1) can emit straight into a packed stream (pack_place).
#include <cooperative_groups.h>

#include <cstdlib>
#include <type_traits>

#include "codec_math.cuh"
#include "device_ctx.h"
#include "kv_codec.h"

namespace cg = cooperative_groups;

namespace speckv {

namespace {

#ifndef SPECKV_KW
#define SPECKV_KW 16
#endif
constexpr int kW = SPECKV_KW;           // warps (= regions) per CTA
constexpr int kThreadsF = kW * 32;
constexpr int kCtasPerSm = 48 / kW;     // 48 warps per SM: 40 registers per thread, <= 227 KiB of tiles
constexpr int kRegion = 2048;           // elements / pairs per region
constexpr int kIters = 8;               // 256 per warp iteration, 8 per lane
constexpr int kRegionBytes = 4096;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxR = 128;              // regions per group, at most

constexpr int kEarlyFlushIter = 3;      // compress: the pairs of iterations 0..3 leave while 4..7 are emitted (+0.6 %)
constexpr int kPadBytes = 512;          // staging slack in front of every region tile (in-place emission)
constexpr int kBlockBytes = kPadBytes + kRegionBytes;

struct FastSmem {
    alignas(128) uint8_t tile[kW][kBlockBytes];   // [pad][4 KiB region]; outputs are staged in place, 16 B..512 B behind the reads
    alignas(8) unsigned long long mbar[kW];
    alignas(8) unsigned long long xmbar[3];   // cluster groups: one per exchange round, completed by the peers' st.async bytes
    // exchange words of ALL regions of the group (every region pushes its word into every CTA of the
    // cluster), indexed by region for cluster groups and by warp for groups inside one CTA
    uint32_t xa[kMaxR];   // region max bits | head count + flags | sum of counts
    uint32_t xb[kMaxR];   // sum of value*count + flags
    uint32_t xc[kMaxR];   // second round of xa (no reuse hazard between rounds)
    uint32_t stash[kW];   // long-run groups: first | (last + 1) << 12 of the region's natural heads, between the two passes
};

// ---- PTX helpers ------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// mbarrier used by this CTA only (bulk-TMA completion): the async proxy must see the initialisation
__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// mbarrier that peer CTAs complete (st.async): the initialisation is released to the cluster
__device__ __forceinline__ void mbar_init_cluster(uint32_t a, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t a, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
// one bulk-TMA copy global -> shared, completion counted in bytes on the mbarrier
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(mbar)
                 : "memory");
}
// Wait for a phase of an mbarrier.  try_wait blocks in hardware for a bounded time (the hint, in ns,
// is an upper bound the hardware may shorten), so the loop rarely spins; measured against plain
// try_wait, try_wait + nanosleep and test_wait + back-off: no difference within 1 %.
__device__ __forceinline__ void mbar_wait(uint32_t a, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(a),
        "r"(parity), "r"(0x989680u)
        : "memory");
}
// one step of an inclusive warp scan: v += (value of lane - o), for the lanes that have such a lane
__device__ __forceinline__ uint32_t scan_step(uint32_t v, int o) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .b32 t;\n"
        "shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n"
        "@p add.u32 %0, %0, t;\n"
        "}"
        : "+r"(v)
        : "r"(o));
    return v;
}
__device__ __forceinline__ uint32_t warp_scan_inclusive(uint32_t v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) v = scan_step(v, o);
    return v;
}
// address of the same shared-memory variable in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t a, uint32_t rank) {
    uint32_t r;
    asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
// asynchronous 4-byte store into a peer CTA's shared memory; the peer's mbarrier counts the bytes
__device__ __forceinline__ void st_async_u32(uint32_t dst, uint32_t v, uint32_t mbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.u32 [%0], %1, [%2];" ::"r"(dst), "r"(v),
                 "r"(mbar)
                 : "memory");
}
__device__ __forceinline__ uint4 lds128(const void* p) { return *reinterpret_cast<const uint4*>(p); }

template <typename T> __device__ __forceinline__ void unpack8(const uint4& raw, float (&x)[8]);
template <> __device__ __forceinline__ void unpack8<__half>(const uint4& raw, float (&x)[8]) {
    const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 f = __half22float2(h[i]);
        x[2 * i] = f.x;
        x[2 * i + 1] = f.y;
    }
}
template <> __device__ __forceinline__ void unpack8<__nv_bfloat16>(const uint4& raw, float (&x)[8]) {
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        x[2 * i] = __uint_as_float(w[i] << 16);
        x[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}

// |x| max of 8 packed elements folded into a packed running max (NaN operands are dropped)
template <typename T> struct Pack2;
template <> struct Pack2<__half> { using type = __half2; };
template <> struct Pack2<__nv_bfloat16> { using type = __nv_bfloat162; };

template <typename T>
__device__ __forceinline__ typename Pack2<T>::type absmax8(typename Pack2<T>::type m, const uint4& raw) {
    using P = typename Pack2<T>::type;
    const P* h = reinterpret_cast<const P*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) m = __hmax2(m, __habs2(h[i]));
    return m;
}
__device__ __forceinline__ float pack_max_to_float(__half2 m) { return fmaxf(__low2float(m), __high2float(m)); }
__device__ __forceinline__ float pack_max_to_float(__nv_bfloat162 m) { return fmaxf(__low2float(m), __high2float(m)); }

template <typename T> __device__ __forceinline__ uint32_t pack2_out(float a, float b);
template <> __device__ __forceinline__ uint32_t pack2_out<__half>(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
template <> __device__ __forceinline__ uint32_t pack2_out<__nv_bfloat16>(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
template <typename T> __device__ __forceinline__ uint16_t out_bits(float a) {
    T h = narrow<T>(a);
    return *reinterpret_cast<uint16_t*>(&h);
}

// Cluster groups exchange their region words without cluster barriers: every region stores its word
// into every CTA of the cluster with st.async, which also credits 4 bytes to an mbarrier in the
// receiving CTA; a CTA's warps wait on their own mbarrier until all R words (R * 4 bytes per array)
// have landed.  One split cluster barrier at kernel start (arrive after the mbarriers are armed,
// wait just before the first remote store) makes sure a peer's shared memory is only written once
// that CTA runs and has armed its mbarriers; by then the peers have long arrived.  The arrive is
// relaxed: fence.mbarrier_init.release.cluster (in mbar_init_cluster) is what publishes the mbarriers.
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// arm the exchange mbarriers of this CTA (one thread), `words` arrays of R words in round 0
template <int R>
__device__ __forceinline__ void exchange_init(FastSmem& sm, int words0, int words1, int words2 = 0) {
    if (R > kW) {
        if (threadIdx.x < 32) {
            // ptxas turns the initialisation into a warp-uniform operation (executed once for warp 0) while the
            // expect_tx stays with thread 0: the __syncwarp in between states their order explicitly
            if (threadIdx.x == 0) {   // one release fence for all of them
                const int n = words2 ? 3 : 2;
                for (int i = 0; i < n; ++i)
                    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&sm.xmbar[i])), "r"(1u) : "memory");
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            }
            __syncwarp();
            if (threadIdx.x == 0) {
                mbar_expect_tx(smem_u32(&sm.xmbar[0]), (uint32_t)(R * 4 * words0));
                if (words1) mbar_expect_tx(smem_u32(&sm.xmbar[1]), (uint32_t)(R * 4 * words1));
                if (words2) mbar_expect_tx(smem_u32(&sm.xmbar[2]), (uint32_t)(R * 4 * words2));   // only long-run groups complete it
            }
        }
        cluster_arrive();
    }
}

// Exchange between the regions of a group.  publish(): the region's lane 0 stores its word into the
// group's array (groups inside one CTA), or lanes 0..C-1 send it to the C CTAs of the cluster.
// group_sync() then waits until every region's word is there; every warp reads the words locally:
// `before` = sum over lower-indexed regions, `total`, `mx` = max.
template <int R>
__device__ __forceinline__ void group_publish(FastSmem& sm, uint32_t* arr, int round, int warp, int lane, int ridx,
                                              uint32_t v) {
    if (R <= kW) {
        if (lane == 0) arr[warp] = v;
    } else {
        constexpr int C = R / kW;
        if (lane < C)
            st_async_u32(mapa_u32(smem_u32(arr + ridx), (uint32_t)lane), v,
                         mapa_u32(smem_u32(&sm.xmbar[round]), (uint32_t)lane));
    }
}

template <int R>
__device__ __forceinline__ void group_sync(FastSmem& sm, int round) {
    if (R == 1) __syncwarp();
    else if (R <= kW) __syncthreads();
    else mbar_wait(smem_u32(&sm.xmbar[round]), 0);
}

// Synchronisation of a round that only SOME groups of a CTA run (the long-run exchange): groups smaller than a CTA
// use a named barrier of their own (ids 1 .. 8, R * 32 threads) instead of __syncthreads.
template <int R>
__device__ __forceinline__ void group_sync_own(FastSmem& sm, int round, int warp) {
    if (R == 1) __syncwarp();
    else if (R < kW) asm volatile("bar.sync %0, %1;" ::"r"(1 + warp / R), "r"(R * 32) : "memory");
    else if (R == kW) __syncthreads();
    else mbar_wait(smem_u32(&sm.xmbar[round]), 0);
}

template <int R>
__device__ __forceinline__ void group_reduce(const uint32_t* arr, int warp, int lane, int ridx, uint32_t& before,
                                             uint32_t& total, uint32_t& mx) {
    if (R == 1) {
        before = 0;
        total = mx = arr[warp];
        return;
    }
    const int base = R <= kW ? (warp / R) * R : 0;
    uint32_t b = 0, t = 0, m = 0;
#pragma unroll
    for (int i = 0; i < (R + 31) / 32; ++i) {
        const int j = i * 32 + lane;
        if (j < R) {
            const uint32_t v = arr[base + j];
            t += v;
            m = max(m, v);
            if (j < ridx) b += v;
        }
    }
    before = __reduce_add_sync(kFull, b);
    total = __reduce_add_sync(kFull, t);
    mx = __reduce_max_sync(kFull, m);
}

__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts16(uint32_t a, uint32_t v) {
    asm volatile("st.shared.b16 [%0], %1;" ::"r"(a), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ uint4 lds128s(uint32_t a) {
    uint4 r;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(a));
    return r;
}
__device__ __forceinline__ uint32_t lds16s(uint32_t a) {
    unsigned short r;
    asm volatile("ld.shared.b16 %0, [%1];" : "=h"(r) : "r"(a));
    return r;
}

// Store n (<= 8, or <= 9 with w4) consecutive 16-bit units held in w0..w3 (w4) at a 2-byte aligned
// shared address.  `n_full` is the register capacity (8 or 9 units); n is n_full or n_full - 1.
__device__ __forceinline__ void store_units8(uint32_t a, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, int n) {
    if ((a & 2u) == 0) {
        sts32(a, w0);
        sts32(a + 4, w1);
        sts32(a + 8, w2);
        if (n == 8) sts32(a + 12, w3);
        else sts16(a + 12, w3);
    } else {
        sts16(a, w0);
        sts32(a + 2, __byte_perm(w0, w1, 0x5432));
        sts32(a + 6, __byte_perm(w1, w2, 0x5432));
        sts32(a + 10, __byte_perm(w2, w3, 0x5432));
        if (n == 8) sts16(a + 14, w3 >> 16);
    }
}
__device__ __forceinline__ void store_units9(uint32_t a, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t w4,
                                             int n) {
    if ((a & 2u) == 0) {
        sts32(a, w0);
        sts32(a + 4, w1);
        sts32(a + 8, w2);
        sts32(a + 12, w3);
        if (n == 9) sts16(a + 16, w4);
    } else {
        sts16(a, w0);
        sts32(a + 2, __byte_perm(w0, w1, 0x5432));
        sts32(a + 6, __byte_perm(w1, w2, 0x5432));
        sts32(a + 10, __byte_perm(w2, w3, 0x5432));
        if (n == 9) sts32(a + 14, __byte_perm(w3, w4, 0x5432));
        else sts16(a + 14, w3 >> 16);
    }
}

// Copy the staged 16-bit units [lo, hi) (indices in the group's output stream) to global memory.
// Unit i lives at shared address sbase + 2*i and at global address gout + 2*i; both are congruent
// mod 16, so the whole vectors in between move with one bulk-TMA store (cp.async.bulk.global.shared::cta;
// measured +7 % compress / +12 % decompress over per-lane 128-bit LDS + STG); the ragged first/last
// vectors (shared with the neighbouring regions' streams) are written in 2-byte pieces, one per lane.
// bulk part only, units [a, b) with a and b multiples of 8 (used for an early partial flush)
__device__ __forceinline__ void flush_bulk(uint32_t sbase, uint8_t* gout, int a, int b, int lane) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0 && b > a) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gout + 2 * (size_t)a),
                     "r"(sbase + 2u * (uint32_t)a), "r"((uint32_t)(b - a) << 1)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
}
__device__ __forceinline__ void flush_region(uint32_t sbase, uint8_t* gout, int lo, int hi, int lane, int done = 0) {
    if (hi <= lo) return;
    int lo_al = min((lo + 7) & ~7, hi);
    const int hi_al = max(hi & ~7, lo_al);
    const int first_al = lo_al;
    lo_al = max(lo_al, min(done, hi_al));   // units [first_al, done) already left with an earlier bulk store
    // the aligned middle leaves with ONE bulk-TMA store issued by lane 0 (no per-vector LDS + STG); the
    // staged pairs were written through the generic proxy, so every lane fences them to the async proxy first
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    const uint32_t bytes = (uint32_t)(hi_al - lo_al) << 1;
    if (lane == 0 && bytes) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gout + 2 * (size_t)lo_al),
                     "r"(sbase + 2u * (uint32_t)lo_al), "r"(bytes)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    int i = lo + lane;
    if (i < first_al) *reinterpret_cast<uint16_t*>(gout + ((size_t)i << 1)) = (uint16_t)lds16s(sbase + ((uint32_t)i << 1));
    i = hi_al + lane;
    if (i < hi) *reinterpret_cast<uint16_t*>(gout + ((size_t)i << 1)) = (uint16_t)lds16s(sbase + ((uint32_t)i << 1));
    // the tile must stay allocated until the copy engine has read it: lane 0 keeps the CTA alive
    if (lane == 0 && (bytes || done)) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// ===================================================================================
// compress: groups with long runs
// ===================================================================================
// A lane chunk without any run boundary (9+ equal deltas: constant stretches, zero tails of partially filled blocks)
// takes its group off the 7-or-8-pairs-per-lane path.  Everything such a group needs follows from one quantity per
// chunk: nb, the position of the last NATURAL head (delta[p] != delta[p-1]) before the chunk.
//   * forced heads (the 255 cap, cache_engine.cpp:223): positions nb + 255 k that are not natural heads; a chunk of 8
//     holds at most one, and only before its first natural head;
//   * a head h closes a run that started at the previous emitted head nb + 255 * floor((h - 1 - nb) / 255).
// nb is an exclusive max-scan of head positions: warp shuffles inside an iteration, a warp-uniform carry across
// iterations, and across regions the exchange of (first, last) natural head per region.  A region counts its natural
// and "interior" forced heads (those after its first natural head) itself; the forced heads in the stretch before the
// first natural head of a region depend on lower regions and are derived by every region for all lower regions from
// the exchanged words (long_reduce).  The kernel reaches all of this through two calls that are deliberately NOT
// inlined (long_first_pass, long_path): inlined, the long-run code costs the common path 1 - 5 % (round 1: 5 %, the
// round-2 routines: 1 %).  Regions of such a group that hold no long run themselves take the common emission
// (emit_common) from inside long_path, with the pair offset the exchange gives them.
__device__ __forceinline__ uint32_t head_mask8(uint32_t nz0, uint32_t nz1) {   // bit j = position j of the chunk starts a run
    const uint32_t lo = (((nz0 >> 7) & 0x01010101u) * 0x01020408u) >> 24;
    const uint32_t hi = (((nz1 >> 7) & 0x01010101u) * 0x01020408u) >> 24;
    return (lo & 0xfu) | ((hi & 0xfu) << 4);
}
// inclusive max-scan over the lanes (values >= -1)
__device__ __forceinline__ int warp_scan_max(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, v, o);
        if (lane >= o) v = max(v, t);
    }
    return v;
}
// x / 255 for any 32-bit x
__device__ __forceinline__ uint32_t div255(uint32_t x) { return __umulhi(x, 0x80808081u) >> 7; }

// Selector table of the head-stationary emission: nibble i of entry m = position of the i-th set bit of m (0 beyond
// popc(m)), so that two byte permutes bring the values (and the positions) of a chunk's heads to the front.  It lives
// in global memory (1 KiB, L1-resident): the lanes index it with different masks, which a __constant__ bank would serialise.
struct HeadSelTable {
    uint32_t v[256];
    constexpr HeadSelTable() : v() {
        for (int m = 0; m < 256; ++m) {
            uint32_t sel = 0;
            int n = 0;
            for (int j = 0; j < 8; ++j)
                if ((m >> j) & 1) sel |= (uint32_t)j << (4 * n++);
            v[m] = sel;
        }
    }
};
__device__ const HeadSelTable kHeadSel = HeadSelTable();

// First pass over a region of a long-run group (phase 2a parked {dsh0, dsh1, nz0, nz1} per lane and iteration).  Per
// chunk: the head mask m (8 bits) and nb, the last natural head before the chunk INSIDE the region -- "the nearest lower
// lane with a head" is one ballot + one shuffle, the carry across iterations is warp-uniform.  Both are cached in the
// chunk's own slot (word 2 = m | (nb_rel + 1) << 8; 0 = none yet in this region) for the emission pass.  Counts the
// interior forced heads (the 255 cap, positions nb + 255 t inside a chunk's leading stretch) and leaves
// first | (last + 1) << 12 of the region's natural heads in *stash (first = 2048, last + 1 = 0 when there is none).
__device__ __forceinline__ uint32_t long_first_pass_body(uint8_t* reg, int lane, uint32_t* stash, bool zero_tail) {
    const unsigned lt = (1u << lane) - 1u;
    uint32_t forced_acc = 0;
    int reg_last = -1, reg_first = 2048;
    for (int k = 0; k < kIters; ++k) {
        if (k == 1 && zero_tail) {
            // a zero region (phase 2a wrote its slots behind iteration 0 as zeros): every chunk from here on is head-less
            // with the same nb, and the forced heads among positions [256, 2048) are the multiples of 255 in
            // [256 - nb, 2048 - nb) -- closed form instead of seven more iterations
            const uint32_t w2 = (uint32_t)(reg_last + 1) << 8;
#pragma unroll
            for (int kk = 1; kk < kIters; ++kk) *reinterpret_cast<uint32_t*>(reg + kk * 512 + lane * 16 + 8) = w2;
            if (reg_last >= 0 && lane == 0) forced_acc += div255(2047u - (uint32_t)reg_last) - div255(255u - (uint32_t)reg_last);
            break;
        }
        uint8_t* slot = reg + k * 512 + lane * 16;
        const uint2 e = *reinterpret_cast<const uint2*>(slot + 8);
        const uint32_t m = head_mask8(e.x, e.y);
        const unsigned bal = __ballot_sync(kFull, m != 0u);
        const int c = k * 256 + lane * 8;
        const int own_last = c + 31 - __clz((int)m);
        const unsigned pl = bal & lt;
        const int t = __shfl_sync(kFull, own_last, pl ? 31 - __clz((int)pl) : 0);
        const int nb = pl ? t : reg_last;
        const int lead_len = m ? __ffs((int)m) - 1 : 8;
        if (nb >= 0) {
            const uint32_t d = (uint32_t)(c - nb);   // >= 1
            forced_acc += div255(d + (uint32_t)lead_len - 1u) - div255(d - 1u);   // multiples of 255 in [d, d + lead_len)
        }
        *reinterpret_cast<uint32_t*>(slot + 8) = m | ((uint32_t)(nb + 1) << 8);
        if (bal) {
            if (reg_first == 2048) reg_first = __shfl_sync(kFull, c + lead_len, __ffs((int)bal) - 1);
            reg_last = __shfl_sync(kFull, own_last, 31 - __clz((int)bal));
        }
    }
    if (lane == 0) *stash = (uint32_t)reg_first | ((uint32_t)(reg_last + 1) << 12);
    return __reduce_add_sync(kFull, forced_acc);
}
#ifdef SPECKV_LONG_INLINE
#define SPECKV_LONG_ATTR __forceinline__
#else
#define SPECKV_LONG_ATTR __noinline__
#endif
// the kernel body calls it out of line (inlined there, the long-run code costs the common path 5 %)
__device__ SPECKV_LONG_ATTR uint32_t long_first_pass(uint8_t* reg, int lane, uint32_t* stash, bool zero_tail) {
    return long_first_pass_body(reg, lane, stash, zero_tail);
}

// Round-2 reduce of a group with long runs.  A: interior head count (low 20 bits) per region, B: first | (last + 1) << 12.
// Gives the number of pairs emitted by lower regions and nb_in, the group position of the last natural head before
// this region (-1 for region 0).
template <int R>
__device__ __forceinline__ void long_reduce(const uint32_t* A, const uint32_t* B, int warp, int lane, int ridx,
                                            uint32_t& h_before, int& nb_in) {
    const int base = R <= kW ? (warp / R) * R : 0;
    int carry = -1;          // last natural head over the regions of earlier blocks of 32
    uint32_t before = 0;
    int mine = -1;
#pragma unroll
    for (int i = 0; i < (R + 31) / 32; ++i) {
        const int j = i * 32 + lane;
        const bool valid = j < R;
        const uint32_t a = valid ? (A[base + j] & 0xfffffu) : 0u;
        const uint32_t b = valid ? B[base + j] : 2048u;
        const int first = (int)(b & 0xfffu), lastp1 = (int)((b >> 12) & 0xfffu);
        const int lastg = lastp1 ? j * kRegion + lastp1 - 1 : -1;
        const int incl = warp_scan_max(lastg, lane);
        const int excl = __shfl_up_sync(kFull, incl, 1);
        const int nb = lane == 0 ? carry : max(carry, excl);
        uint32_t lead = 0;
        if (valid && j > 0 && nb >= 0) {
            const int a0 = j * kRegion, bnd = a0 + min(first, kRegion);
            lead = (uint32_t)((bnd - 1 - nb) / 255 - (a0 - 1 - nb) / 255);
        }
        if (valid && j < ridx) before += a + lead;
        if (valid && j == ridx) mine = nb;
        carry = max(carry, __shfl_sync(kFull, incl, 31));
    }
    h_before = __reduce_add_sync(kFull, before);
    nb_in = (int)__reduce_max_sync(kFull, (unsigned)(mine + 1)) - 1;
}

// one 16-bit unit to shared memory under a predicate (stays a predicated STS: no branch)
__device__ __forceinline__ void sts16_if(uint32_t a, uint32_t v, bool on) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.u32 p, %2, 0;\n"
        "@p st.shared.b16 [%0], %1;\n"
        "}" ::"r"(a),
        "h"((unsigned short)v), "r"((uint32_t)on)
        : "memory");
}

// Ragged groups (the filled prefix of a block): v = elements of a lane chunk that lie before the group's end.
// mask_tail8 zeroes the elements at or past it (they take no part in the max); tail_heads8 makes every position at
// or past it a run head, so the run open at the end closes there with the reference's last pair and every pair
// behind it is dropped at emission -- the head count up to the end, and with it every offset, stays the reference's.
__device__ __forceinline__ uint4 mask_tail8(uint4 raw, int v) {
    if (v >= 8) return raw;
    uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) w[i] &= (2 * i < v ? 0x0000ffffu : 0u) | (2 * i + 1 < v ? 0xffff0000u : 0u);
    return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ uint2 tail_heads8(int v) {
    const int a = min(max(v, 0), 4), b = min(max(v - 4, 0), 4);
    return make_uint2(a == 4 ? 0u : 0x80808080u << (8 * a), b == 4 ? 0u : 0x80808080u << (8 * b));
}

// Phase 2b of a region of a group with long runs.  Per chunk (from the slot: dsh0, dsh1 and the first pass's m | nb):
// the previous emitted head before the chunk is nb + 255 * floor((c - 1 - nb) / 255); a forced head falls into the
// chunk's leading stretch when the next multiple does; then the chunk's natural heads, head-stationary: the selector
// table compacts their values and positions, the counts are the byte-wise differences of the positions (the first one
// reaches back to the previous emitted head).  Iterations without any head are skipped after the vote.
//
// The body has NO lane-divergent branch: every store is predicated.  A first version stored the units through an
// if / else ladder on (alignment, count) inside "if (m)"; on the B200 the lanes that skipped the block were then seen
// to run on without the others (the shuffle that fetches lane 31's running count returned the reader's own value, the
// loop's uniform counter was stepped by both halves) although the block ends in the compiler's reconvergence point --
// bit-exact with printf in the loop, wrong without.  With at most the warp-uniform "continue" left, there is nothing
// to reconverge.
// Returns the pair index after the region; prev_end = the last emitted head before the end of the region.
__device__ __forceinline__ int long_emit(const uint8_t* reg, uint32_t sbase, int lane, int rstart, int pidx, int nb_in,
                                         int& prev_end) {
    int last_emitted = 0;
    for (int k = 0; k < kIters; ++k) {
        const uint4 st = lds128(reg + k * 512 + lane * 16);
        __syncwarp();   // every lane has read its slot before any pair of this iteration lands on it
        const int c = rstart + k * 256 + lane * 8;
        const uint32_t m = st.z & 0xffu, nbr1 = st.z >> 8;
        const int nb = nbr1 ? rstart + (int)nbr1 - 1 : nb_in;   // group position of the last natural head before the chunk
        const int lead_len = m ? __ffs((int)m) - 1 : 8;
        int prev = 0, pf = 0x7fffffff;
        if (nb >= 0) {
            prev = nb + 255 * (int)div255((uint32_t)(c - 1 - nb));   // previous emitted head (natural or forced), <= c - 1
            pf = prev + 255;                                        // the next forced head, >= c
        }
        const bool forced = pf < c + lead_len;
        const int nn = __popc(m), n = nn + (forced ? 1 : 0);
        last_emitted = m ? c + 31 - __clz((int)m) : (forced ? pf : prev);
        if (__ballot_sync(kFull, m != 0u) == 0u) {
            // no natural head in the whole iteration (inside a long run): only the cap's forced heads, at most two lanes
            const unsigned fb = __ballot_sync(kFull, forced);
            if (fb == 0u) continue;
            const uint32_t fj0 = (uint32_t)(pf - c);
            sts16_if(sbase + 2u * (uint32_t)(pidx + __popc(fb & ((1u << lane) - 1u))),
                     ((((fj0 & 4u) ? st.y : st.x) >> (8u * (fj0 & 3u))) & 0xffu) | 0xff00u, forced);
            pidx += __popc(fb);
            continue;
        }
        const int inc = (int)warp_scan_inclusive((uint32_t)n);
        const int idx = pidx + inc - n;
        // the forced pair closes 255 positions of the run whose delta is delta[pf - 1] (byte pf - c of the shifted deltas)
        const uint32_t fj = (uint32_t)(pf - c);   // 0 .. 7 when forced
        sts16_if(sbase + 2u * (uint32_t)idx, ((((fj & 4u) ? st.y : st.x) >> (8u * (fj & 3u))) & 0xffu) | 0xff00u, forced);
        if (forced) prev = pf;
        const uint32_t a = sbase + 2u * (uint32_t)(idx + (forced ? 1 : 0));
        const uint32_t sel = __ldg(&kHeadSel.v[m]);
        const uint32_t v0 = __byte_perm(st.x, st.y, sel & 0xffffu), v1 = __byte_perm(st.x, st.y, sel >> 16);
        const uint32_t p0 = __byte_perm(0x03020100u, 0x07060504u, sel & 0xffffu);
        const uint32_t p1 = __byte_perm(0x03020100u, 0x07060504u, sel >> 16);
        // counts: position differences; bytes beyond the last head are garbage (borrows only travel upwards)
        const uint32_t c0 = p0 - (p0 << 8) + (uint32_t)(c - prev), c1 = p1 - __funnelshift_l(p0, p1, 8);
        const uint32_t w0 = __byte_perm(v0, c0, 0x5140), w1 = __byte_perm(v0, c0, 0x7362);
        const uint32_t w2 = __byte_perm(v1, c1, 0x5140), w3 = __byte_perm(v1, c1, 0x7362);
        sts16_if(a, w0, nn > 0);
        sts16_if(a + 2, w0 >> 16, nn > 1);
        sts16_if(a + 4, w1, nn > 2);
        sts16_if(a + 6, w1 >> 16, nn > 3);
        sts16_if(a + 8, w2, nn > 4);
        sts16_if(a + 10, w2 >> 16, nn > 5);
        sts16_if(a + 12, w3, nn > 6);
        sts16_if(a + 14, w3 >> 16, nn > 7);
        pidx += __shfl_sync(kFull, inc, 31);
    }
    prev_end = __shfl_sync(kFull, last_emitted, 31);
    return pidx;
}

// ===================================================================================
// compress: phase 2b, the common emission (every run shorter than 9: no chunk without a head)
// ===================================================================================
// `last`: the region that holds the group's last element.  A ragged group has `lim` elements in this region (>= 2048:
// all).  Its iterations wholly past them are skipped; the positions past them inside the last iteration run (`cut`)
// are forced heads, so the last `cut` pairs staged are dropped (the pair the head at the group's end emits is the
// reference's last one, cache_engine.cpp:235-236).
template <int R, bool RAGGED>
__device__ __forceinline__ void emit_common(uint8_t* reg, uint32_t reg_s, int lane, unsigned lt_mask, int ridx, uint32_t h_before,
                                            uint32_t halo_tail, uint32_t carry_d1, float s, uint8_t* gout, float* scale_out,
                                            uint32_t* comp_out, bool last, int lim) {
    const int k_end = RAGGED ? (min(lim, kRegion) + 255) >> 8 : kIters;
    const int cut = RAGGED ? k_end * 256 - min(lim, kRegion) : 0;
    // ---- 2b. emit: a head at position p closes the previous run -> pair (delta[p-1], p - previous head).
    //          Pairs are staged IN PLACE (behind the slots still to be read) at the alignment they
    //          will have in global memory, then the region goes out with one bulk-TMA store.
    // Region 0 starts at pair index -1: the head at position 0 closes nothing, so its "pair" is
    // staged in the pad in front of the tile and never flushed.
    int pidx = (int)h_before - 1;
    const int p0 = max(pidx, 0);                         // first real pair index of this region
    const uint32_t sbase = reg_s - 16u - 2u * (uint32_t)(p0 & ~7);   // pair i is staged at sbase + 2*i
    // tail = distance from the end of a lane chunk back to its last head; the next chunk's first
    // pair closes a run of that length (+ its own offset)
    uint32_t carry_tail = halo_tail;
    const int src_lane = (lane + 31) & 31;
#ifndef SPECKV_UNROLL_2B
#define SPECKV_UNROLL_2B 8
#endif
    int done = 0;   // units below this index already left with an early bulk store
    constexpr int kUnroll2b = SPECKV_UNROLL_2B;   // full unrolling measured 2.4 % faster than 2; fetching slot k + 1 early: slower
#pragma unroll kUnroll2b
    for (int k = 0; k < kIters; ++k) {
        if (RAGGED && k >= k_end) break;
        const uint4 st = lds128(reg + k * 512 + lane * 16);
        __syncwarp();   // every lane has read its slot before any pair of this iteration lands on it
        const uint32_t dsh0 = st.x, dsh1 = st.y;
        const uint32_t nz0 = st.z, nz1 = st.w;
        const uint32_t hw0 = ~nz0 & 0x80808080u, hw1 = ~nz1 & 0x80808080u;   // "holes": positions that continue a run
        const int nhole = __popc(hw0) + __popc(hw1);
        if (!__any_sync(kFull, nhole > 1)) {
            // ---- common case: every lane emits 8 pairs, or 7 (one position continues a run) ----
            // with at most one hole the run open at the end of the chunk is 1 or 2 positions long
            const uint32_t rt = __shfl_sync(kFull, 1u + (hw1 >> 31), src_lane);
            const uint32_t lf = lane == 0 ? carry_tail : rt;   // distance back to the previous head
            carry_tail = rt;
            const unsigned bal = __ballot_sync(kFull, nhole != 0);
            const int idx = pidx + 8 * lane - __popc(bal & lt_mask);
            // Branch-free hole deletion.  u = 1 << (8 * hole byte) in its word, 0 without a hole.
            // counts: lf for the first unit, 1 elsewhere; once the hole unit is gone the unit that
            // takes its index has absorbed the hole's position: +1 at that index (lf + 1 at index 0).
            const uint32_t u0 = hw0 >> 7, u1 = hw1 >> 7;
            const uint32_t c0 = (0x01010100u | lf) + u0, c1 = 0x01010101u + u1;
            // values: bytes below the hole stay, bytes from the hole on move down by one
            const uint32_t keep0 = u0 - 1u;                    // all ones when the hole is not in word 0
            const uint32_t keep1 = u0 ? 0u : u1 - 1u;
            const uint32_t sh0 = __funnelshift_r(dsh0, dsh1, 8), sh1 = dsh1 >> 8;
            const uint32_t v0 = (dsh0 & keep0) | (sh0 & ~keep0), v1 = (dsh1 & keep1) | (sh1 & ~keep1);
            const uint32_t w0 = __byte_perm(v0, c0, 0x5140), w1 = __byte_perm(v0, c0, 0x7362);
            const uint32_t w2 = __byte_perm(v1, c1, 0x5140), w3 = __byte_perm(v1, c1, 0x7362);
            store_units8(sbase + 2u * (uint32_t)idx, w0, w1, w2, w3, 8 - nhole);
            pidx += 256 - __popc(bal);
        } else {
            // ---- some lane has two or more continuing positions: scan + one store per head ----
            const uint32_t tail = nz1 ? ((uint32_t)__clz((int)nz1) >> 3) + 1u : ((uint32_t)__clz((int)nz0) >> 3) + 5u;
            const uint32_t rt = __shfl_sync(kFull, tail, src_lane);
            const uint32_t lf = lane == 0 ? carry_tail : rt;
            carry_tail = rt;
            const int n = 8 - nhole;
            const int inc = (int)warp_scan_inclusive((uint32_t)n);
            int idx = pidx + inc - n;
            uint32_t run = lf;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t v = (j < 4 ? dsh0 >> (8 * j) : dsh1 >> (8 * (j - 4))) & 0xffu;
                const uint32_t isz = (j < 4 ? nz0 >> (8 * j) : nz1 >> (8 * (j - 4))) & 0x80u;
                if (isz) {
                    sts16(sbase + 2u * (uint32_t)idx, v | (run << 8));
                    ++idx;
                    run = 1;
                } else {
                    ++run;
                }
            }
            pidx += __shfl_sync(kFull, inc, 31);
        }
        if (k == kEarlyFlushIter && (!RAGGED || lim >= kRegion / 2)) {
            // the pairs staged so far are final: the whole vectors among them leave now, overlapping the rest
            // (ragged: only when every head so far lies before the group's end)
            done = max(pidx & ~7, (p0 + 7) & ~7);
            flush_bulk(sbase, gout, (p0 + 7) & ~7, done, lane);
        }
    }
    if (last) {
        // the run still open at the end of the group (cache_engine.cpp:235-236)
        if (lane == 0) {
            const uint32_t cnt = carry_tail;
            sts16(sbase + 2u * (uint32_t)pidx, (carry_d1 >> 24) | (cnt << 8));
            *scale_out = s;
            *comp_out = 2u * (uint32_t)(pidx + 1 - (RAGGED ? cut : 0));
        }
        ++pidx;
    }
    __syncwarp();
    flush_region(sbase, gout, p0, RAGGED && last ? pidx - cut : pidx, lane, done);
}

// Phase 2b of a group with long runs, as ONE routine outside the kernel body (the common path keeps its code and
// register allocation): a third exchange (first / last natural head per region), offsets from long_reduce, every
// iteration through the general routine, the final pair, the flush.
// Ragged groups: regions past the end (!live) take part in the exchange only.
template <int R, bool RAGGED>
__device__ SPECKV_LONG_ATTR void long_path(FastSmem& sm, uint8_t* reg, uint32_t reg_s, int warp, int lane, int ridx, bool longr,
                                       uint32_t carry_d1, uint32_t halo_tail, float s, uint8_t* gout, float* scale_out,
                                       uint32_t* comp_out, bool live, bool last, int lim) {
    constexpr uint32_t G = (uint32_t)R * kRegion;
    const int cut = RAGGED ? kRegion - min(lim, kRegion) : 0;   // forced heads behind the group's end in this region
    // regions with a head-less chunk ran the first pass in phase 2a (their interior forced heads went into round 2 and
    // first | last natural head into the stash); in the others these two sit in the first and the last lane chunk
    uint32_t stash_w;
    if (RAGGED && !live) {
        stash_w = (uint32_t)kRegion;   // no natural head
    } else if (!longr) {
        uint2 e = make_uint2(0u, 0u);   // lane 0 and lane 31 read the flags they parked themselves
        if (lane == 0) e = *reinterpret_cast<const uint2*>(reg + 8);
        else if (lane == 31) e = *reinterpret_cast<const uint2*>(reg + (kIters - 1) * 512 + 31 * 16 + 8);
        const uint32_t m = head_mask8(e.x, e.y);
        const int reg_first = __shfl_sync(kFull, __ffs((int)m) - 1, 0);
        const int reg_last = __shfl_sync(kFull, (kIters - 1) * 256 + 31 * 8 + 31 - __clz((int)m), 31);
        stash_w = (uint32_t)reg_first | ((uint32_t)(reg_last + 1) << 12);
    } else {
        __syncwarp();
        stash_w = sm.stash[warp];
    }
    group_publish<R>(sm, sm.xb, 2, warp, lane, ridx, stash_w);
    group_sync_own<R>(sm, 2, warp);
    uint32_t hb;
    int nb_in;
    long_reduce<R>(sm.xc, sm.xb, warp, lane, ridx, hb, nb_in);
    if (RAGGED && !live) return;
    if (!longr) {
        // A region WITHOUT a head-less chunk and with a head among the 8 positions in front of it: no run of 16 or more
        // touches it, so no forced head falls into it -- the common emission, behind the pairs of the lower regions
        // (dense regions of a partially filled block, the noise around one constant stretch).
        emit_common<R, RAGGED>(reg, reg_s, lane, (1u << lane) - 1u, ridx, hb, halo_tail, carry_d1, s, gout, scale_out, comp_out,
                               last, lim);
        return;
    }
    int pl = (int)hb - 1;
    const int pl0 = max(pl, 0);
    const uint32_t sb = reg_s - 16u - 2u * (uint32_t)(pl0 & ~7);
    int prev_end;
    pl = long_emit(reg, sb, lane, ridx * kRegion, pl, nb_in, prev_end);
    if (last) {
        if (lane == 0) {
            const int end = RAGGED ? (ridx + 1) * kRegion : (int)G;
            sts16(sb + 2u * (uint32_t)pl, (carry_d1 >> 24) | ((uint32_t)(end - prev_end) << 8));   // cache_engine.cpp:235-236
            *scale_out = s;
            *comp_out = 2u * (uint32_t)(pl + 1 - (RAGGED ? cut : 0));
        }
        ++pl;
    }
    __syncwarp();
    flush_region(sb, gout, pl0, RAGGED && last ? pl - cut : pl, lane);
}

// ===================================================================================
// compress: packed emission (page groups, R = 1)
// ===================================================================================
// The tier's offload wants the payloads back to back (what crosses PCIe), not one worst-case slot per group.  A
// group's size is known once its run heads are counted (2 bytes per head), i.e. before any pair is staged, so the
// compress kernel can place the groups itself: the 16 groups of a CTA are scanned in shared memory, the CTAs chain
// through one status word each (decoupled look-back: [2-bit state | 62-bit bytes], state 1 = this CTA's total,
// 2 = inclusive prefix; warp 0 polls 32 predecessors per step).  CTAs start in blockIdx order and a CTA waits only
// for lower ones, so the chain always advances.  A group left to the generic kernel reserves a whole slot.
enum : unsigned long long { kPackAgg = 1ull << 62, kPackIncl = 2ull << 62, kPackErr = 1ull << 61, kPackVal = (1ull << 61) - 1 };

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// byte offset of this warp's group in the packed stream; called by ALL warps of the CTA (two block barriers).
// A predecessor that never shows up (it cannot happen while CTAs start in blockIdx order) must not hang the device:
// a poll gives up after ~10 s and marks its word; the mark travels down the chain and the stream's total becomes
// ~0, which the host treats as a failed launch.
__device__ __noinline__ unsigned long long pack_place(FastSmem& sm, const PackOut& pk, uint32_t my_bytes, int warp, int lane) {
    if (lane == 0) sm.xb[warp] = my_bytes;
    __syncthreads();
    const uint32_t v = lane < kW ? sm.xb[lane] : 0u;
    const uint32_t incl = warp_scan_inclusive(v);
    const uint32_t before = __shfl_sync(kFull, incl - v, warp);
    const uint32_t cta_total = __shfl_sync(kFull, incl, kW - 1);
    if (warp == 0) {
        unsigned long long prefix = 0;
        bool err = false;
        volatile unsigned long long* status = pk.status;
        const uint32_t b = blockIdx.x;
        if (b != 0) {
            if (lane == 0) status[b] = kPackAgg | cta_total;
            long long base = (long long)b - 1;
            for (;;) {
                const long long idx = base - lane;
                unsigned long long w;
                uint32_t polls = 0;
                do {
                    w = idx >= 0 ? status[idx] : kPackIncl;   // in front of CTA 0: prefix 0
                    if (++polls == (1u << 23)) w = kPackIncl | kPackErr;   // ~1 us per poll
                } while (__any_sync(kFull, (w >> 62) == 0ull));
                const unsigned incl_mask = __ballot_sync(kFull, (w >> 62) == 2ull);
                const unsigned long long val = w & kPackVal;
                const int first = incl_mask ? __ffs((int)incl_mask) - 1 : 31;   // the nearest predecessor that knows its prefix
                err |= __any_sync(kFull, lane <= first && (w & kPackErr) != 0ull);
                prefix += warp_sum_u64(lane <= first ? val : 0ull);
                if (incl_mask) break;   // everything behind it is included
                base -= 32;
            }
        }
        if (lane == 0) {
            status[b] = kPackIncl | (err ? kPackErr : 0ull) | ((prefix + cta_total) & kPackVal);
            sm.xc[kW] = (uint32_t)prefix;
            sm.xc[kW + 1] = (uint32_t)(prefix >> 32);
            if (b == gridDim.x - 1) *pk.total = err ? ~0ull : prefix + cta_total;
        }
    }
    __syncthreads();
    return ((unsigned long long)sm.xc[kW] | ((unsigned long long)sm.xc[kW + 1] << 32)) + before;
}

// ===================================================================================
// compress
// ===================================================================================
// RAGGED: group g is the first n = a.group_length(g, G) elements of its block.  Regions at or past n are neither
// loaded nor emitted but still take part in every exchange (a cluster CTA stays until its peers' words have landed);
// the region holding element n - 1 masks its tail out of the max, forces run heads from n on and ends the group.
template <typename T, int R, bool PACKED = false, bool RAGGED = false>
__global__ void __launch_bounds__(kThreadsF, kCtasPerSm)
compress_fast_kernel(const __grid_constant__ CodecArgs a, uint32_t* __restrict__ needs_generic, const PackOut pk) {
    static_assert(!PACKED || R == 1, "packed emission is built for page groups");
    static_assert(!(PACKED && RAGGED), "ragged groups use the slot form");
    extern __shared__ __align__(128) uint8_t smem_raw[];
    FastSmem& sm = *reinterpret_cast<FastSmem*>(smem_raw);
    constexpr int C = R > kW ? R / kW : 1;        // CTAs per group (cluster size)
    constexpr int GPC = R >= kW ? 1 : kW / R;     // groups per CTA
    constexpr uint32_t G = (uint32_t)R * kRegion;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    uint32_t g;
    int ridx;
    if (R >= kW) {
        const unsigned crank = C > 1 ? cg::this_cluster().block_rank() : 0u;
        g = blockIdx.x / C;
        ridx = (int)crank * kW + warp;
    } else {
        g = blockIdx.x * GPC + warp / R;
        ridx = warp % R;
    }
    const bool active = g < a.n_groups;
    const uint32_t n_len = (RAGGED && active) ? a.group_length(g, G) : G;
    const int lim = (int)n_len - ridx * kRegion;                 // elements of this region inside the group (>= 2048: all)
    const bool live = active && (!RAGGED || lim > 0);
    const T* in = static_cast<const T*>(a.in);
    // a group past the end has no elem_index entry to read: its (never loaded) address stays block g
    const T* rin = (active ? a.elem_block(in, g, G) : in + (size_t)g * G) + (size_t)ridx * kRegion;
    uint8_t* reg = sm.tile[warp] + kPadBytes;
    const uint32_t reg_s = smem_u32(reg);
    const uint32_t mb = smem_u32(&sm.mbar[warp]);

    // ---- 0. one bulk-TMA copy per region (issued before anything else: the exchange set-up hides behind it) ----
    if (lane == 0) {
        mbar_init(mb, 1);
        if (live) {
            const uint32_t bytes = RAGGED ? (uint32_t)min(kRegionBytes, ((lim + 7) & ~7) * 2) : (uint32_t)kRegionBytes;
            mbar_expect_tx(mb, bytes);
            tma_load_1d(reg_s, rin, bytes, mb);
        }
    }
    __syncwarp();
    exchange_init<R>(sm, 1, 1, 1);
    // halo: the 16 elements in front of the region, fetched now so that the latency hides behind phase 1
    T halo_x = narrow<T>(0.0f);
    if (live && ridx > 0 && lane < 16) halo_x = __ldg(rin + lane - 16);

    // ---- 1. region max-abs, then the group max over its R regions -------------------------------
    float m = 0.0f;
    if (live) {
        mbar_wait(mb, 0);
        const uint32_t z = 0u;
        typename Pack2<T>::type pm = *reinterpret_cast<const typename Pack2<T>::type*>(&z);
#pragma unroll
        for (int k = 0; k < kIters; ++k) {
            if (RAGGED && k * 256 >= lim) break;
            const uint4 raw = lds128(reg + k * 512 + lane * 16);
            pm = absmax8<T>(pm, (RAGGED && lim < kRegion) ? mask_tail8(raw, lim - (k * 256 + lane * 8)) : raw);
        }
        // non-negative floats order like their bit patterns: one integer warp reduction
        m = __uint_as_float(__reduce_max_sync(kFull, __float_as_uint(pack_max_to_float(pm))));
    }
    // only +-0 and NaN in this region (a ragged group's boundary region keeps the general path: its tail is heads)
    const bool zero_region = live && __float_as_uint(m) == 0u && (!RAGGED || lim >= kRegion);
    if (C > 1) cluster_wait();   // all CTAs of the cluster are running: their shared memory may be written
    group_publish<R>(sm, sm.xa, 0, warp, lane, ridx, __float_as_uint(m));   // non-negative floats order like their bits
    group_sync<R>(sm, 0);
    uint32_t t0, t1, gmax_bits;
    group_reduce<R>(sm.xa, warp, lane, ridx, t0, t1, gmax_bits);
    const float gmax = __uint_as_float(gmax_bits);
    const bool fast = fast_quant_ok<T>(gmax);
    // max / 127 (the reference), or max for the clamped scheme.  For the groups this kernel encodes itself (fast) the
    // IEEE division by 127 is the two-operation form RN(m * r127 + RN(m * d127)) of codec_math.cuh: exact for every
    // fp16 value and every bf16 value >= 2^-118 (oracle/verify_fastdiv.c, "scale"), a dozen instructions shorter
    const float s = scheme_max_scale(a.scheme) ? (gmax > 0.0f ? gmax : 1.0f)
                                    : (fast ? __fmaf_rn(gmax, __uint_as_float(0x3c010204u), __fmul_rn(gmax, __uint_as_float(0x2e010204u)))
                                            : scale_from_max(gmax));
    // a group whose max-abs is 0 (zeros, possibly NaNs: cache_engine.cpp:176-179 skips them and the cast maps
    // them to code 0) has the closed-form payload [0][255] x floor(G/255) + [0][G%255]: no second read
    const bool zero_group = active && gmax_bits == 0u;
    float r, rl;
    recip_hi_lo(s, r, rl);

    // ---- 2a. quantise, delta, run-boundary flags; results parked in the lane's own 16-byte slot ----
    // slot = { dsh0, dsh1 : deltas shifted by one element (byte j = delta[pos_j - 1]),
    //          nz0,  nz1  : bit 7 of byte j set iff position j starts a run (delta[j] != delta[j-1]) }
    uint32_t heads = 0;
    bool cplx = !fast && !zero_group;
    bool longr = false;       // a chunk (or the halo) without any run boundary: the group takes the long-run path
    uint32_t carry_d1 = 0, halo_tail = 1u;   // halo_tail: distance from the region's first position back to the last head before it
    if (live && fast) {
        if (ridx > 0) {
            // halo: the 16 elements before the region give the last code, the last delta and the
            // run boundaries among the last 4 positions before the region (all local, no neighbour needed)
            uint32_t qh = 0;
            if (lane < 16) qh = quantize_fast(widen<T>(halo_x), r, rl);
            const uint32_t qp = __shfl_up_sync(kFull, qh, 1);
            const uint32_t dh = (qh - qp) & 0xffu;
            const uint32_t dp = __shfl_up_sync(kFull, dh, 1);
            const unsigned chg = __ballot_sync(kFull, lane >= 8 && lane < 16 && dh != dp) >> 8;   // bit i: position i - 8 starts a run
            halo_tail = chg ? (uint32_t)__clz((int)chg) - 23u : 9u;
            carry_d1 = __shfl_sync(kFull, (qh & 0xffu) | (dh << 24), 15);   // code in byte 0, delta in byte 3
            if (chg == 0) longr = true;   // a run of 9+ equal deltas reaches the region edge
        }
        const int src_lane = (lane + 31) & 31;
        uint32_t half_k = HalfConst<T>::k;
        asm volatile("" : "+r"(half_k));   // keep it in a register: LOP3 takes only one immediate
#pragma unroll
        for (int k = 0; k < kIters; ++k) {
            if (k == 1 && zero_region) {
                // A region of zeros (and NaNs: code 0 as well) inside a non-zero group -- the unused tail of a
                // partially filled block.  Its codes are all 0, so behind the first chunks (iteration 0 settles the
                // hand-over from the previous region) every delta, shifted delta and boundary flag is 0: the slots
                // are written without quantising anything.  The carries keep iteration 0's values (0 as well).
#pragma unroll
                for (int kk = 1; kk < kIters; ++kk) *reinterpret_cast<uint4*>(reg + kk * 512 + lane * 16) = make_uint4(0u, 0u, 0u, 0u);
                longr = true;   // head-less chunks
                break;
            }
            uint8_t* slot = reg + k * 512 + lane * 16;
            if (RAGGED && k * 256 >= lim) {
                // wholly past the group's end: every position a head (only the long-run routines read these slots).
                // The head at the group's end itself (lane 0 of the first such iteration) closes the reference's last
                // run, whose value long_emit takes from shifted-delta byte 0: delta[n - 1], which lane 0's carry holds
                // in byte 3 (lane 31 of the previous iteration).  Every later pair is dropped.
                const uint32_t d_end = (lane == 0 && k * 256 == lim) ? carry_d1 >> 24 : 0u;
                *reinterpret_cast<uint4*>(slot) = make_uint4(d_end, 0u, 0x80808080u, 0x80808080u);
                heads += 8;
                continue;
            }
            const uint4 raw = lds128(slot);
            float x[8];
            unpack8<T>(raw, x);
            uint32_t q[8];
            const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
                quantize_fast_pair_i<T>(rw[j], x[2 * j], x[2 * j + 1], r, rl, half_k, q[2 * j], q[2 * j + 1]);
            // what the position in front of the chunk hands over -- its code (byte 0) and its delta (byte 3) -- comes in
            // ONE shuffle: from lane - 1, or (lane 0) from lane 31 of the previous iteration
            uint32_t d[8];
#pragma unroll
            for (int j = 1; j < 8; ++j) d[j] = q[j] - q[j - 1];
            const uint32_t rx = __shfl_sync(kFull, __byte_perm(q[7], d[7], 0x4000), src_lane);
            const uint32_t px = lane == 0 ? carry_d1 : rx;
            carry_d1 = rx;
            d[0] = q[0] - px;
            const uint32_t d0 = __byte_perm(__byte_perm(d[0], d[1], 0x0040), __byte_perm(d[2], d[3], 0x0040), 0x5410);
            const uint32_t d1 = __byte_perm(__byte_perm(d[4], d[5], 0x0040), __byte_perm(d[6], d[7], 0x0040), 0x5410);
            const uint32_t dsh0 = __byte_perm(px, d0, 0x6543);
            const uint32_t dsh1 = __byte_perm(d0, d1, 0x6543);
            const uint32_t x0 = d0 ^ dsh0, x1 = d1 ^ dsh1;
            uint32_t nz0 = (((x0 & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x0) & 0x80808080u;
            uint32_t nz1 = (((x1 & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x1) & 0x80808080u;
            if (ridx == 0 && k == 0 && lane == 0) nz0 |= 0x80u;   // position 0 always starts a run
            if (RAGGED && lim < kRegion) {   // warp-uniform: the boundary region only
                const uint2 th = tail_heads8(lim - (k * 256 + lane * 8));
                nz0 |= th.x;
                nz1 |= th.y;
            }
            const int nh = __popc(nz0) + __popc(nz1);
            longr |= (nh == 0);                                   // a run of 9+ equal deltas: long-run path
            heads += nh;
            *reinterpret_cast<uint4*>(slot) = make_uint4(dsh0, dsh1, nz0, nz1);
        }
        // after the loop lane 0's carries hold lane 31's last code word; make them warp-uniform
        carry_d1 = __shfl_sync(kFull, carry_d1, 0);
        heads = __reduce_add_sync(kFull, heads);
    }
    longr = __any_sync(kFull, longr);
    if (longr && live && fast) heads += long_first_pass(reg, lane, &sm.stash[warp], zero_region);   // forced heads behind the region's first natural head
    // one word per region: head count (natural + interior forced, <= 2056) in the low 20 bits, "has long runs" counted
    // above.  "Needs the generic kernel" (a scale outside the fast quantiser's domain) follows from the group max,
    // which every region already has: no exchange needed.
    group_publish<R>(sm, sm.xc, 1, warp, lane, ridx, live ? (heads | (longr ? (1u << 20) : 0u)) : 0u);
    group_sync<R>(sm, 1);
    uint32_t h_before, h_total;
    group_reduce<R>(sm.xc, warp, lane, ridx, h_before, h_total, t0);
    const bool any_cplx = cplx;
    const bool any_long = (h_total >> 20) != 0;
    h_before &= 0xfffffu;
    size_t out_off = 0;   // packed emission only; the slot form derives its address where it is used (no live range across the exchange)
    if constexpr (PACKED) {
        // bytes of this group: 2 per run head (the head at position 0 emits nothing, the open run at the end one pair),
        // the closed form of a zero group, a whole slot for a group the generic kernel will encode
        constexpr uint32_t zfull = G / 255u, zrem = G % 255u, znp = zfull + (zrem ? 1u : 0u);
        uint32_t my = 0;
        if (active) my = cplx ? (uint32_t)a.slot_bytes : (zero_group ? 2u * znp : 2u * (h_total & 0xfffffu));
        out_off = (size_t)pack_place(sm, pk, (my + 15u) & ~15u, warp, lane);
        if (active && lane == 0) pk.offsets[g] = out_off;
    }
    if (!active) return;
    if (ridx == 0 && lane == 0) {
        needs_generic[g] = any_cplx ? 1u : 0u;
        if (any_cplx) a.comp_bytes[g] = gmax_bits;   // hand the group max to the generic kernel: it skips its own max pass
    }
    if (any_cplx) return;
    if (zero_group) {
        if (ridx == 0) {
            const uint32_t full = n_len / 255u, rem = n_len % 255u, npairs = full + (rem ? 1u : 0u);
            uint16_t* go = reinterpret_cast<uint16_t*>(static_cast<uint8_t*>(a.payload) + (PACKED ? out_off : (size_t)g * a.slot_bytes));
            for (uint32_t i = lane; i < npairs; i += 32u) go[i] = i < full ? (uint16_t)0xff00u : (uint16_t)(rem << 8);
            if (lane == 0) {
                a.scales[g] = s;   // 1.0f
                a.comp_bytes[g] = 2u * npairs;
            }
        }
        return;
    }

    uint8_t* gout = static_cast<uint8_t*>(a.payload) + (PACKED ? out_off : (size_t)g * a.slot_bytes);
    const bool last = RAGGED ? lim > 0 && lim <= kRegion : ridx == R - 1;   // the region holds the group's last element
    if (any_long) {   // groups with long runs: everything else happens in long_path (not inlined)
        long_path<R, RAGGED>(sm, reg, reg_s, warp, lane, ridx, longr, carry_d1, halo_tail, s, gout, a.scales + g, a.comp_bytes + g,
                             live, last, lim);
        return;
    }
    if (RAGGED && !live) return;

    emit_common<R, RAGGED>(reg, reg_s, lane, (1u << lane) - 1u, ridx, h_before, halo_tail, carry_d1, s, gout, a.scales + g, a.comp_bytes + g,
                           last, lim);
}

// ===================================================================================
// decompress
// ===================================================================================
// Rare-path helpers of phase A, out of line (the kernel keeps its registers): the index of the first pair of the
// region's zero-valued tail (0 = every value is zero; pairs past the payload were blanked before), and the element
// count of that tail while its pairs are blanked in the tile (count 0 emits nothing in the expansion).
__device__ __noinline__ uint32_t zero_tail_start(const uint8_t* reg, int lane) {
    int last_nz = -1;
#pragma unroll
    for (int k = 0; k < kIters; ++k) {
        const uint4 w = lds128(reg + k * 512 + lane * 16);
        const uint32_t va = __byte_perm(w.x, w.y, 0x6420), vb = __byte_perm(w.z, w.w, 0x6420);
        const uint32_t za = (((va & 0x7f7f7f7fu) + 0x7f7f7f7fu) | va) & 0x80808080u;
        const uint32_t zb = (((vb & 0x7f7f7f7fu) + 0x7f7f7f7fu) | vb) & 0x80808080u;
        const int pbase = k * 256 + lane * 8;
        if (zb) last_nz = pbase + 4 + ((31 - __clz((int)zb)) >> 3);
        else if (za) last_nz = pbase + ((31 - __clz((int)za)) >> 3);
    }
    return __reduce_max_sync(kFull, (unsigned)(last_nz + 1));
}
__device__ __noinline__ uint32_t zero_tail_blank(uint8_t* reg, int lane, uint32_t np, uint32_t t_first) {
    uint32_t tsum = 0;
    for (int k = 0; k < kIters; ++k) {
        const int pbase = k * 256 + lane * 8;
        if (pbase + 8 > (int)t_first && pbase < (int)np) {
            uint32_t* slot = reinterpret_cast<uint32_t*>(reg + k * 512 + lane * 16);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                uint32_t w = slot[i];
                if (pbase + 2 * i >= (int)t_first) {
                    tsum += (w >> 8) & 0xffu;
                    w &= 0xffff0000u;
                }
                if (pbase + 2 * i + 1 >= (int)t_first) {
                    tsum += w >> 24;
                    w &= 0x0000ffffu;
                }
                slot[i] = w;
            }
        }
    }
    return __reduce_add_sync(kFull, tsum);
}

template <typename T, int R>
__global__ void __launch_bounds__(kThreadsF, kCtasPerSm)
decompress_fast_kernel(const __grid_constant__ CodecArgs a, const DecodeScratch scr) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    FastSmem& sm = *reinterpret_cast<FastSmem*>(smem_raw);
    constexpr int C = R > kW ? R / kW : 1;
    constexpr int GPC = R >= kW ? 1 : kW / R;
    constexpr uint32_t G = (uint32_t)R * kRegion;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1u;

    uint32_t g;
    int ridx;
    if (R >= kW) {
        const unsigned crank = C > 1 ? cg::this_cluster().block_rank() : 0u;
        g = blockIdx.x / C;
        ridx = (int)crank * kW + warp;
    } else {
        g = blockIdx.x * GPC + warp / R;
        ridx = warp % R;
    }
    // the request count may live on the device (prefetch requests routed by a kernel): the grid covers the
    // capacity n_groups, groups at or above the count only clear their flag for the generic second pass
    const bool in_grid = g < a.n_groups;
    const bool active = in_grid && g < a.live_groups();
    uint8_t* reg = sm.tile[warp] + kPadBytes;
    const uint32_t reg_s = smem_u32(reg);
    const uint32_t mb = smem_u32(&sm.mbar[warp]);

    // pairs of this region: [ridx * 2048, ridx * 2048 + np)
    uint32_t np = 0;
    float s = 1.0f;
    bool cplx = false;
    const uint8_t* rp = nullptr;   // the region's pairs
    if (active) {
        const uint32_t gi = a.stored_block(g);
        const uint32_t cb = __ldg(a.comp_bytes + gi);
        uint32_t npairs = cb >> 1;                            // a trailing odd byte is ignored (:245-247)
        if ((size_t)cb > a.slot_bytes) cplx = true;           // malformed: leave it to the generic kernel's clamping
        npairs = min(npairs, (uint32_t)(R * kRegion));
        const uint32_t first = (uint32_t)ridx * kRegion;
        np = npairs > first ? min(npairs - first, (uint32_t)kRegion) : 0u;
        s = __ldg(a.scales + gi);
        cplx |= scale_is_special(s);
        rp = a.block_payload(gi) + (size_t)ridx * kRegionBytes;
    }

    if (lane == 0) {
        mbar_init(mb, 1);
        if (np > 0) {
            const uint32_t bytes = ((np * 2u) + 15u) & ~15u;
            mbar_expect_tx(mb, bytes);
            tma_load_1d(reg_s, rp, bytes, mb);
        }
    }
    __syncwarp();
    exchange_init<R>(sm, 2, 0);

    // ---- dequantiser choice (while the tile is in flight).  y = ((float) q / 127.0f) * s costs four operations per
    // element (codec_math.cuh); q * RN(s / 127) costs two and, after the final rounding to fp16 / bf16, gives the same
    // bits for almost every scale.  "Almost" is settled exactly: there are only 256 codes, so the regions of a group
    // check them all against the reference form for this group's scale (256 / R codes per region) and the group
    // takes the short form only if every code agrees -- the output stays bit-identical either way (decompress +3 %;
    // more than 99 % of the scales qualify).
    constexpr bool kTryShort = R >= 8;   // at most one code per lane to check; smaller groups keep the reference form
    const float kq = __fdiv_rn(s, 127.0f);
    bool deq_differs = !kTryShort;
    if (kTryShort && active && !cplx) {
        constexpr int CPR = 256 / R;   // codes checked by each region
        for (int c = lane; c < CPR; c += 32) {
            const uint32_t code = (uint32_t)(ridx * CPR + c);
            const float qf = (float)(int)(int8_t)code;
            deq_differs |= out_bits<T>(dequantize(code, s)) != out_bits<T>(__fmul_rn(qf, kq));
        }
        deq_differs = __any_sync(kFull, deq_differs);
    }

    // ---- the expansion loop (phase C), defined here because one-region groups run it without phase A ----
    uint32_t ecur = 0;                                     // next element index to produce
    uint32_t qcur = 0;                                     // code of element ecur - 1
    uint32_t sbase = reg_s - (uint32_t)kPadBytes;          // element i is staged at sbase + 2*i
    uint32_t rd_s = reg_s + 16u * (uint32_t)lane;          // this lane's slot of the current iteration
#ifndef SPECKV_UNROLL_C
#define SPECKV_UNROLL_C 1
#endif
    constexpr int kUnrollC = SPECKV_UNROLL_C;
    // kShort: the verified two-operation dequantiser.  kSingle: no phase A ran -- pairs past the end of the payload are
    // blanked here and the staging bound is enforced on the fly; returns false when the region has to go to the
    // generic kernel instead (it expands beyond what in-place staging can hold).
    auto expand = [&](auto short_tag, auto single_tag) -> bool {
    constexpr bool kShort = decltype(short_tag)::value;
    constexpr bool kSingle = decltype(single_tag)::value;
    auto deq = [&](uint32_t code) -> float {
        return kShort ? __fmul_rn((float)(int)(int8_t)code, kq) : dequantize(code, s);
    };
#pragma unroll kUnrollC
    for (uint32_t pk = 0; pk < np; pk += 256u, rd_s += 512u) {
        uint4 w = lds128s(rd_s);
        __syncwarp();
        if (kSingle && pk + 256u > np) {   // the last, partial iteration: blank the pairs past the end (count 0 emits nothing)
            const int nv = min(max((int)np - (int)pk - lane * 8, 0), 8);
            uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (2 * i >= nv) ww[i] = 0u;
                else if (2 * i + 1 >= nv) ww[i] &= 0x0000ffffu;
            }
            w = make_uint4(ww[0], ww[1], ww[2], ww[3]);
        }
        const uint32_t va = __byte_perm(w.x, w.y, 0x6420), ca = __byte_perm(w.x, w.y, 0x7531);
        const uint32_t vb = __byte_perm(w.z, w.w, 0x6420), cb = __byte_perm(w.z, w.w, 0x7531);
        // counts: c - 1 is 0 for a count of 1 and 1 for a count of 2; a count of 0 borrows and any
        // other count leaves higher bits, so "every count is 1 or 2" is one mask test
        const uint32_t ta = ca - 0x01010101u, tb = cb - 0x01010101u;   // byte j = 1 iff count j is 2
        const bool small = ((ta | tb) & 0xfefefefeu) == 0;
        const int ntwo = __popc(ta) + __popc(tb);
        const bool slow = __any_sync(kFull, !small || ntwo > 1);
        const uint32_t sl = __dp4a(vb, cb, __dp4a(va, ca, 0u));
        if (!slow) {
            // every lane: 8 pairs -> 8 or 9 elements
            const unsigned bal = __ballot_sync(kFull, ntwo != 0);
            // in-place staging: the elements of this iteration must end before the slots still to be read (an
            // earlier iteration with long counts may have used up the slack)
            if (kSingle && ecur + 256u + (uint32_t)__popc(bal) > pk + 512u - 8u) return false;
            const uint32_t idx = ecur + 8u * lane + __popc(bal & lt_mask);
            const uint32_t inc = warp_scan_inclusive(sl);
            const uint32_t tot = __shfl_sync(kFull, inc, 31);
            const uint32_t qb = qcur + inc - sl;
            // Branch-free duplication of the value whose count is 2 (ta / tb hold 1 << (8 * its byte)):
            // bytes up to and including it stay, the bytes above move up by one; the ninth value is
            // byte 7 either way (it is only stored when there was a duplicate).
            const uint32_t keep0 = (ta << 8) - 1u;                  // all ones when the pair is not in word a
            const uint32_t keep1 = ta ? 0u : (tb << 8) - 1u;
            const uint32_t up0 = va << 8, up1 = __funnelshift_l(va, vb, 8);
            const uint32_t v0 = (va & keep0) | (up0 & ~keep0), v1 = (vb & keep1) | (up1 & ~keep1);
            const uint32_t v2 = vb >> 24;
            // codes = running byte sums: dp4a against 0x01, 0x0101, ... adds the first 1..4 bytes
            float y[9];
            const uint32_t q4 = __dp4a(v0, 0x01010101u, qb);
            y[0] = deq(__dp4a(v0, 0x00000001u, qb));
            y[1] = deq(__dp4a(v0, 0x00000101u, qb));
            y[2] = deq(__dp4a(v0, 0x00010101u, qb));
            y[3] = deq(q4);
            y[4] = deq(__dp4a(v1, 0x00000001u, q4));
            y[5] = deq(__dp4a(v1, 0x00000101u, q4));
            y[6] = deq(__dp4a(v1, 0x00010101u, q4));
            const uint32_t q8 = __dp4a(v1, 0x01010101u, q4);
            y[7] = deq(q8);
            y[8] = deq(q8 + v2);
            store_units9(sbase + 2u * idx, pack2_out<T>(y[0], y[1]), pack2_out<T>(y[2], y[3]), pack2_out<T>(y[4], y[5]),
                         pack2_out<T>(y[6], y[7]), pack2_out<T>(y[8], 0.0f), 8 + ntwo);
            ecur += 256u + __popc(bal);
            qcur = (qcur + tot) & 0xffu;
        } else {
            // any counts: exclusive scan of (elements, code advance), then per-pair loops
            const uint32_t cl = __dp4a(cb, 0x01010101u, __dp4a(ca, 0x01010101u, 0u));
            const uint32_t inc = warp_scan_inclusive(cl | (sl << 24));
            const uint32_t tot = __shfl_sync(kFull, inc, 31);
            const uint32_t excl = inc - (cl | (sl << 24));
            // in-place staging: the elements of this iteration must end before the slots still to be read
            if (kSingle && ecur + (tot & 0xffffffu) > pk + 512u - 8u) return false;
            uint32_t p = ecur + (excl & 0xffffffu);
            uint32_t q = qcur + (excl >> 24);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t v = (j < 4 ? va >> (8 * j) : vb >> (8 * (j - 4))) & 0xffu;
                const uint32_t c = (j < 4 ? ca >> (8 * j) : cb >> (8 * (j - 4))) & 0xffu;
                for (uint32_t t = 0; t < c; ++t) {
                    q += v;
                    sts16(sbase + 2u * (p + t), out_bits<T>(dequantize(q & 0xffu, s)));
                }
                p += c;
            }
            ecur += tot & 0xffffffu;
            qcur = (qcur + (tot >> 24)) & 0xffu;
        }
    }
    return true;
    };

    // ---- one-region groups (4 KiB pages): a single pass.  The region starts at element 0 with code 0, so nothing has
    // to be known from phase A; its bookkeeping (decoded length, "expands too far for in-place staging", "longer than the
    // group") falls out of the expansion itself.  Tiny payloads (zero pages are 9 pairs) keep the two-phase path, which
    // decodes them as a constant fill.
    if (R == 1 && active && !cplx && np > 64) {
        mbar_wait(mb, 0);
        const bool ok = expand(std::false_type{}, std::true_type{}) && ecur <= G;
        if (lane == 0) {
            scr.flags[g] = ok ? 0u : 1u;
            if (a.out_elems && ok) a.out_elems[g] = ecur;
        }
        if (!ok) return;
        __syncwarp();
        flush_region(sbase, reinterpret_cast<uint8_t*>(a.elem_block(static_cast<T*>(a.out), g, G)), 0, (int)ecur, lane);
        return;
    }

    // ---- A. region totals: elements produced (sum of counts) and code advance (sum of value*count) ----
    uint32_t csum = 0, ssum = 0, nnz = 0;
    bool fill = false;   // region decoded as a constant fill (all pair values zero) instead of through the staging area
    bool runs = false;   // region expands beyond what in-place staging holds: the group goes to the run-expansion path
    uint32_t tail_elems = 0, np_front = 0;   // split region: np_front pairs expanded in place, then tail_elems elements of fill
    if (np > 0) {
        mbar_wait(mb, 0);
#pragma unroll
        for (int k = 0; k < kIters; ++k) {
            const int pbase = k * 256 + lane * 8;
            const int nv = min(max((int)np - pbase, 0), 8);
            uint8_t* slot = reg + k * 512 + lane * 16;
            uint4 w = lds128(slot);
            if (nv < 8) {   // blank the pairs past the end of the payload (count 0 emits nothing)
                uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (2 * i >= nv) ww[i] = 0u;
                    else if (2 * i + 1 >= nv) ww[i] &= 0x0000ffffu;
                }
                w = make_uint4(ww[0], ww[1], ww[2], ww[3]);
                *reinterpret_cast<uint4*>(slot) = w;
            }
            const uint32_t va = __byte_perm(w.x, w.y, 0x6420), ca = __byte_perm(w.x, w.y, 0x7531);
            const uint32_t vb = __byte_perm(w.z, w.w, 0x6420), cb = __byte_perm(w.z, w.w, 0x7531);
            if (__all_sync(kFull, ca == 0x01010101u && cb == 0x01010101u)) {   // one element per pair
                csum += 8u;
                nnz += 8u;
                ssum = __dp4a(vb, 0x01010101u, __dp4a(va, 0x01010101u, ssum));
            } else {
                csum = __dp4a(cb, 0x01010101u, __dp4a(ca, 0x01010101u, csum));
                ssum = __dp4a(vb, cb, __dp4a(va, ca, ssum));
                nnz += __popc((((ca & 0x7f7f7f7fu) + 0x7f7f7f7fu) | ca) & 0x80808080u) +
                       __popc((((cb & 0x7f7f7f7fu) + 0x7f7f7f7fu) | cb) & 0x80808080u);
            }
        }
        csum = __reduce_add_sync(kFull, csum);
        ssum = __reduce_add_sync(kFull, ssum) & 0xffu;
        nnz = __reduce_add_sync(kFull, nnz);
        // in-place staging needs the output stream to stay within kPadBytes of the read position.  A region that
        // expands further is still decoded here when all its pair values are zero (zero blocks, long constant
        // stretches): every element then repeats the code the region starts with, and nothing is staged.
        if (csum - nnz > (uint32_t)(kPadBytes / 2 - 8)) {
            // where the region's last pair with a non-zero value sits: none -> constant fill; otherwise the pairs behind
            // it (value 0: the code stays) are the zero tail of a partially filled block or the end of a long constant
            // stretch -- if the pairs in front of them fit the staging area, they are expanded in place and the tail
            // is written as a fill behind them (split), and the group stays off the run-expansion path
            const uint32_t t_first = zero_tail_start(reg, lane);   // first pair of the zero-valued tail
            fill = t_first == 0u;
            if (!fill) {
                const uint32_t tsum = zero_tail_blank(reg, lane, np, t_first);
                if ((csum - tsum) - t_first <= (uint32_t)(kPadBytes / 2 - 8) && nnz == np) {
                    tail_elems = tsum;
                    np_front = t_first;
                } else {
                    runs = true;
                }
            }
        }
        // a pair with count 0 (never written by the encoder) emits nothing: such payloads keep to the generic kernel,
        // whose tables allow several pairs at one output position
        if (nnz != np) cplx = true;
    }
    if (C > 1) cluster_wait();   // all CTAs of the cluster are running: their shared memory may be written
    group_publish<R>(sm, sm.xa, 0, warp, lane, ridx, min(csum, G + 1u));   // saturated: sums stay < 2^32, "> G" still shows
    // xb: code advance (8 bits; the sum over <= 128 regions stays below bit 16) | "needs the generic kernel" counted
    // in bits 16..23 | "short dequantiser differs" counted in bits 24..30 | bit 31 "needs the run-expansion path" (read
    // from the MAXIMUM over the regions' words; in the sum it only disturbs bit 31, which nobody reads)
    group_publish<R>(sm, sm.xb, 0, warp, lane, ridx,
                     ssum | (cplx ? (1u << 16) : 0u) | (deq_differs ? (1u << 24) : 0u) | (runs ? (1u << 31) : 0u));
    group_sync<R>(sm, 0);
    uint32_t e_before, e_total, q_before, xb_total, xb_max, t0;
    group_reduce<R>(sm.xa, warp, lane, ridx, e_before, e_total, t0);
    group_reduce<R>(sm.xb, warp, lane, ridx, q_before, xb_total, xb_max);
    if (!active) {
        if (in_grid && ridx == 0 && lane == 0) scr.flags[g] = 0u;
        return;
    }
    const bool any_cplx = ((xb_total >> 16) & 0xffu) != 0 || e_total > G;   // output longer than the group: generic kernel clips
    const bool any_runs = !any_cplx && (xb_max >> 31) != 0u;
    const bool short_deq = ((xb_total >> 24) & 0x7fu) == 0;
    if (ridx == 0 && lane == 0) {
        scr.flags[g] = any_cplx ? 1u : (any_runs ? 2u : 0u);
        if (a.out_elems && !any_cplx) a.out_elems[g] = e_total;
    }
    if (any_runs) {
        // hand the group over with what phase A found: where every pairs-region starts in the output and with which
        // code; the second pass expands output region by output region (kv_codec_generic.cu, decode_runs_region)
        if (lane == 0) {
            scr.prefix[(size_t)g * (R + 1) + ridx] = make_uint2(e_before, q_before & 0xffu);
            if (ridx == 0) {
                scr.prefix[(size_t)g * (R + 1) + R] = make_uint2(e_total, 0u);
                scr.list[atomicAdd(scr.counters, 1u)] = g;
            }
        }
        return;
    }
    if (any_cplx || np == 0) return;

    // ---- C. expand in place: element e of run j carries code q_before + ... + v_j * (e - start_j + 1) ----
    uint8_t* gout = reinterpret_cast<uint8_t*>(a.elem_block(static_cast<T*>(a.out), g, G));
    const uint32_t e0 = e_before;
    // constant fill: elements [ea, ea + n) all carry `code` (zero blocks, long runs of one value, zero tails)
    auto fill_const = [&](uint32_t ea, uint32_t n, uint32_t code) {
        const uint32_t e1 = ea + n;
        const uint32_t hb = out_bits<T>(dequantize(code & 0xffu, s));
        const uint32_t w2 = hb | (hb << 16);
        const uint32_t a0 = min((ea + 7u) & ~7u, e1), a1 = max(e1 & ~7u, a0);
        uint16_t* go16 = reinterpret_cast<uint16_t*>(gout);
        if (ea + lane < a0) go16[ea + lane] = (uint16_t)hb;
        if (a1 + lane < e1) go16[a1 + lane] = (uint16_t)hb;
        const uint4 v4 = make_uint4(w2, w2, w2, w2);
        for (uint32_t e = a0 + 8u * lane; e < a1; e += 256u) *reinterpret_cast<uint4*>(go16 + e) = v4;
    };
    if (fill) {
        fill_const(e0, csum, q_before);
        return;
    }
    ecur = e0;
    qcur = q_before & 0xffu;
    sbase = reg_s - (uint32_t)kPadBytes - 2u * (e0 & ~7u);
    if (tail_elems) np = np_front;   // split region: the pairs of the zero-valued tail were blanked in phase A
    if (kTryShort && short_deq) expand(std::integral_constant<bool, kTryShort>{}, std::false_type{});
    else expand(std::false_type{}, std::false_type{});
    __syncwarp();
    flush_region(sbase, gout, (int)e0, (int)ecur, lane);   // (an early partial flush, as in compress, measured slower here)
    if (tail_elems) fill_const(ecur, tail_elems, qcur);     // the tail repeats the code the expansion ended on
}

// ===================================================================================
// codes-only schemes (INT8 and its clamped variant): quantize_to_int8 / dequantize_from_int8 alone
// (cache_engine.cpp:186-196, :275-284).  Compress is the kernel above without its second half: one bulk-TMA load per
// region, region max, one exchange for the group max, eight codes per lane and iteration written in place, one
// bulk-TMA store of the region's 2 KiB.  Decompress has no dependency between regions at all: no cluster, no exchange.
// Algorithmic traffic: 2n + n bytes per group either way.
// ===================================================================================
// RAGGED: group g is the first n = a.group_length(g, G) elements of its block; n codes are written.
template <typename T, int R, bool RAGGED = false>
__global__ void __launch_bounds__(kThreadsF, kCtasPerSm)
compress_codes_fast_kernel(const __grid_constant__ CodecArgs a, uint32_t* __restrict__ needs_generic) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    FastSmem& sm = *reinterpret_cast<FastSmem*>(smem_raw);
    constexpr int C = R > kW ? R / kW : 1;
    constexpr int GPC = R >= kW ? 1 : kW / R;
    constexpr uint32_t G = (uint32_t)R * kRegion;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t g;
    int ridx;
    if (R >= kW) {
        const unsigned crank = C > 1 ? cg::this_cluster().block_rank() : 0u;
        g = blockIdx.x / C;
        ridx = (int)crank * kW + warp;
    } else {
        g = blockIdx.x * GPC + warp / R;
        ridx = warp % R;
    }
    const bool active = g < a.n_groups;
    const uint32_t n_len = (RAGGED && active) ? a.group_length(g, G) : G;
    const int lim = (int)n_len - ridx * kRegion;   // elements of this region inside the group (>= 2048: all)
    const bool live = active && (!RAGGED || lim > 0);
    const T* in = static_cast<const T*>(a.in);
    // a group past the end has no elem_index entry to read: its (never loaded) address stays block g
    const T* rin = (active ? a.elem_block(in, g, G) : in + (size_t)g * G) + (size_t)ridx * kRegion;
    uint8_t* reg = sm.tile[warp] + kPadBytes;
    const uint32_t reg_s = smem_u32(reg);
    const uint32_t mb = smem_u32(&sm.mbar[warp]);
    if (lane == 0) {
        mbar_init(mb, 1);
        if (live) {
            const uint32_t bytes = RAGGED ? (uint32_t)min(kRegionBytes, ((lim + 7) & ~7) * 2) : (uint32_t)kRegionBytes;
            mbar_expect_tx(mb, bytes);
            tma_load_1d(reg_s, rin, bytes, mb);
        }
    }
    __syncwarp();
    exchange_init<R>(sm, 1, 0);
    float m = 0.0f;
    if (live) {
        mbar_wait(mb, 0);
        const uint32_t z = 0u;
        typename Pack2<T>::type pm = *reinterpret_cast<const typename Pack2<T>::type*>(&z);
#pragma unroll
        for (int k = 0; k < kIters; ++k) {
            if (RAGGED && k * 256 >= lim) break;
            const uint4 raw = lds128(reg + k * 512 + lane * 16);
            pm = absmax8<T>(pm, (RAGGED && lim < kRegion) ? mask_tail8(raw, lim - (k * 256 + lane * 8)) : raw);
        }
        m = __uint_as_float(__reduce_max_sync(kFull, __float_as_uint(pack_max_to_float(pm))));
    }
    if (C > 1) cluster_wait();
    group_publish<R>(sm, sm.xa, 0, warp, lane, ridx, __float_as_uint(m));
    group_sync<R>(sm, 0);
    uint32_t t0, t1, gmax_bits;
    group_reduce<R>(sm.xa, warp, lane, ridx, t0, t1, gmax_bits);
    if (!active) return;
    const float gmax = __uint_as_float(gmax_bits);
    const float s = scale_for(gmax, scheme_max_scale(a.scheme));
    const bool zero_group = gmax_bits == 0u;                 // zeros / NaNs only: every code is 0 (scale 1)
    const bool fast = fast_quant_ok<T>(gmax) || zero_group;
    if (ridx == 0 && lane == 0) {
        needs_generic[g] = fast ? 0u : 1u;
        if (!fast) a.comp_bytes[g] = gmax_bits;              // the generic second pass skips its own max pass
    }
    if (!fast) return;
    if (RAGGED && !live) {   // past the end (an empty group: region 0 reports it)
        if (ridx == 0 && lane == 0) {
            a.scales[g] = s;
            a.comp_bytes[g] = 0u;
        }
        return;
    }
    float r, rl;
    recip_hi_lo(s, r, rl);
    uint32_t half_k = HalfConst<T>::k;
    asm volatile("" : "+r"(half_k));
#pragma unroll
    for (int k = 0; k < kIters; ++k) {
        if (RAGGED && k * 256 >= lim) break;
        const uint4 raw = lds128(reg + k * 512 + lane * 16);
        __syncwarp();   // the codes of this iteration land on bytes that iterations <= k read
        float x[8];
        unpack8<T>(raw, x);
        uint32_t q[8];
        const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) quantize_fast_pair_i<T>(rw[j], x[2 * j], x[2 * j + 1], r, rl, half_k, q[2 * j], q[2 * j + 1]);
        const uint32_t c0 = __byte_perm(__byte_perm(q[0], q[1], 0x0040), __byte_perm(q[2], q[3], 0x0040), 0x5410);
        const uint32_t c1 = __byte_perm(__byte_perm(q[4], q[5], 0x0040), __byte_perm(q[6], q[7], 0x0040), 0x5410);
        *reinterpret_cast<uint2*>(reg + k * 256 + lane * 8) = make_uint2(c0, c1);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    // ragged: the codes before the group's end, whole 16-byte vectors in the bulk store, the rest byte by byte
    const uint32_t nb = RAGGED ? (uint32_t)min(lim, kRegion) : (uint32_t)kRegion;
    const uint32_t nb16 = nb & ~15u;
    uint8_t* gout = static_cast<uint8_t*>(a.payload) + (size_t)g * a.slot_bytes + (size_t)ridx * kRegion;
    if (RAGGED && (uint32_t)lane < nb - nb16) gout[nb16 + lane] = reg[nb16 + lane];
    if (lane == 0) {
        if (nb16)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gout), "r"(reg_s), "r"(nb16)
                         : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        if (ridx == 0) {
            a.scales[g] = s;
            a.comp_bytes[g] = n_len;
        }
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

// one warp per region of 2048 codes; scr.regions = R of the group geometry (any value: regions are independent)
template <typename T>
__global__ void __launch_bounds__(kThreadsF, kCtasPerSm)
decompress_codes_fast_kernel(const __grid_constant__ CodecArgs a, const DecodeScratch scr) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    FastSmem& sm = *reinterpret_cast<FastSmem*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t rid = (uint64_t)blockIdx.x * kW + warp;
    const uint32_t g = (uint32_t)(rid / scr.regions), ridx = (uint32_t)(rid % scr.regions);
    const uint32_t G = scr.regions * (uint32_t)kRegion;
    const bool in_grid = g < a.n_groups;
    const bool active = in_grid && g < a.live_groups();
    if (!in_grid) return;
    uint32_t gi = g, n = 0;
    float s = 1.0f;
    bool cplx = false;
    if (active) {
        gi = a.stored_block(g);
        s = __ldg(a.scales + gi);
        // oversized payloads and non-finite scales: the generic kernel's clamping / special values.  A shorter payload
        // (a ragged group) decodes to its comp_bytes elements here; the rest of the destination is left as it is.
        n = __ldg(a.comp_bytes + gi);
        cplx = n > G || (size_t)G > a.slot_bytes || scale_is_special(s);
    }
    if (ridx == 0 && lane == 0) {
        scr.flags[g] = (active && cplx) ? 1u : 0u;
        if (a.out_elems && active && !cplx) a.out_elems[g] = n;
    }
    const uint32_t nr = n > ridx * (uint32_t)kRegion ? min(n - ridx * (uint32_t)kRegion, (uint32_t)kRegion) : 0u;   // codes of this region
    if (!active || cplx || nr == 0) return;
    uint8_t* reg = sm.tile[warp] + kPadBytes;
    const uint32_t reg_s = smem_u32(reg);
    const uint32_t mb = smem_u32(&sm.mbar[warp]);
    const uint8_t* rp = a.block_payload(gi) + (size_t)ridx * kRegion;
    if (lane == 0) {
        mbar_init(mb, 1);
        const uint32_t bytes = (nr + 15u) & ~15u;   // within the slot: slot_bytes >= G
        mbar_expect_tx(mb, bytes);
        tma_load_1d(reg_s + (uint32_t)kRegion, rp, bytes, mb);   // codes in the upper half: expansion runs in place
    }
    __syncwarp();
    mbar_wait(mb, 0);
#pragma unroll
    for (int k = 0; k < kIters; ++k) {
        if ((uint32_t)k * 256u >= nr) break;
        const uint2 c = *reinterpret_cast<const uint2*>(reg + kRegion + k * 256 + lane * 8);
        __syncwarp();   // iteration 7 writes over the codes it reads
        float y[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = dequantize(((j < 4 ? c.x : c.y) >> (8 * (j & 3))) & 0xffu, s);
        *reinterpret_cast<uint4*>(reg + k * 512 + lane * 16) =
            make_uint4(pack2_out<T>(y[0], y[1]), pack2_out<T>(y[2], y[3]), pack2_out<T>(y[4], y[5]), pack2_out<T>(y[6], y[7]));
    }
    T* gout = a.elem_block(static_cast<T*>(a.out), g, G) + (size_t)ridx * kRegion;
    if (nr < (uint32_t)kRegion) {   // the region holding the end of a short payload: exactly nr elements
        __syncwarp();
        flush_region(reg_s, reinterpret_cast<uint8_t*>(gout), 0, (int)nr, lane);
        return;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gout), "r"(reg_s), "r"((uint32_t)kRegionBytes)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
}

// ---- launch -------------------------------------------------------------------------
template <typename... P, typename... Args>
cudaError_t launch_clustered(void (*kernel)(P...), int R, uint32_t n_groups, cudaStream_t st, Args... args) {
    const int C = R > kW ? R / kW : 1;
    const int gpc = R >= kW ? 1 : kW / R;
    const size_t smem = sizeof(FastSmem);
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(R >= kW ? (size_t)n_groups * C : ((size_t)n_groups + gpc - 1) / gpc));
    cfg.blockDim = dim3(kThreadsF);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // Cluster scheduling policy: load balancing measured 2.4 % (compress) / 3.6 % (decompress) faster than the
    // default (= spread) for clusters of 4 at 3 CTAs per SM.  SPECKV_CLUSTER_POLICY=0|1|2 overrides (default, spread, lb).
    static const int policy = [] { const char* e = std::getenv("SPECKV_CLUSTER_POLICY"); return e ? std::atoi(e) : 2; }();
    if (C > 1 && policy) {
        attr[1].id = cudaLaunchAttributeClusterSchedulingPolicyPreference;
        attr[1].val.clusterSchedulingPolicyPreference =
            policy == 1 ? cudaClusterSchedulingPolicySpread : cudaClusterSchedulingPolicyLoadBalancing;
        cfg.numAttrs = 2;
    }
    e = cudaLaunchKernelEx(&cfg, kernel, args...);
    count_launch();
    return e;
}

template <typename T>
cudaError_t compress_fast_t(int R, const CodecArgs& a, uint32_t* flags, cudaStream_t st, unsigned long long* pack_status) {
    const uint32_t n = a.n_groups;
    if (pack_status) {
        if (R != 1 || scheme_is_codes(a.scheme) || !a.pack_offsets || !a.pack_total || a.group_len) return cudaErrorInvalidValue;
        PackOut pk;
        pk.offsets = a.pack_offsets;
        pk.total = a.pack_total;
        pk.status = pack_status;
        return launch_clustered(compress_fast_kernel<T, 1, true>, 1, n, st, a, flags, pk);
    }
    // ragged calls (a.group_len) run their own instantiations: the dense ones keep their code and registers
    if (scheme_is_codes(a.scheme)) {
        switch (R) {
#define SPECKV_CASE(RR) case RR: return a.group_len ? launch_clustered(compress_codes_fast_kernel<T, RR, true>, RR, n, st, a, flags) \
                                                    : launch_clustered(compress_codes_fast_kernel<T, RR>, RR, n, st, a, flags);
            SPECKV_CASE(1) SPECKV_CASE(2) SPECKV_CASE(4) SPECKV_CASE(8) SPECKV_CASE(16) SPECKV_CASE(32) SPECKV_CASE(64) SPECKV_CASE(128)
#undef SPECKV_CASE
            default: return cudaErrorInvalidValue;
        }
    }
    switch (R) {
#define SPECKV_CASE(RR) case RR: return a.group_len ? launch_clustered(compress_fast_kernel<T, RR, false, true>, RR, n, st, a, flags, PackOut{}) \
                                                : launch_clustered(compress_fast_kernel<T, RR>, RR, n, st, a, flags, PackOut{});
        SPECKV_CASE(1) SPECKV_CASE(2) SPECKV_CASE(4) SPECKV_CASE(8) SPECKV_CASE(16) SPECKV_CASE(32) SPECKV_CASE(64) SPECKV_CASE(128)
#undef SPECKV_CASE
        default: return cudaErrorInvalidValue;
    }
}

template <typename T>
cudaError_t decompress_fast_t(int R, const CodecArgs& a, const DecodeScratch& scr, cudaStream_t st) {
    if (scheme_is_codes(a.scheme)) {
        const size_t smem = sizeof(FastSmem);
        cudaError_t e = cudaFuncSetAttribute(decompress_codes_fast_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        const uint64_t regions = (uint64_t)a.n_groups * (uint32_t)R;
        decompress_codes_fast_kernel<T><<<(unsigned)((regions + kW - 1) / kW), kThreadsF, smem, st>>>(a, scr);
        count_launch();
        return cudaGetLastError();
    }
    switch (R) {
#define SPECKV_CASE(RR) case RR: return launch_clustered(decompress_fast_kernel<T, RR>, RR, a.n_groups, st, a, scr);
        SPECKV_CASE(1) SPECKV_CASE(2) SPECKV_CASE(4) SPECKV_CASE(8) SPECKV_CASE(16) SPECKV_CASE(32) SPECKV_CASE(64) SPECKV_CASE(128)
#undef SPECKV_CASE
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace

// regions per group if the tuned kernels cover this geometry, else 0
int fast_regions(const CodecArgs& a, bool decompress) {
    if (!(scheme_is_rle(a.scheme) || scheme_is_codes(a.scheme)) || (a.dtype != DT_F16 && a.dtype != DT_BF16)) return 0;
    if (a.group_elems == 0 || a.group_elems % kRegion) return 0;
    const uint32_t R = a.group_elems / kRegion;
    if (R > 128 || (R & (R - 1))) return 0;
    if (R > (uint32_t)kW * 8) return 0;   // portable cluster size limit (8 CTAs)
    // a cache set: the alignment of its bases and stride, recorded when it was created
    const void* elems = a.cache_bases ? nullptr : decompress ? a.out : a.in;
    if (a.cache_bases && a.set_unaligned) return 0;
    if ((reinterpret_cast<uintptr_t>(elems) | reinterpret_cast<uintptr_t>(a.payload)) & 15) return 0;
    if (a.slot_bytes < (size_t)R * (scheme_is_codes(a.scheme) ? kRegion : kRegionBytes)) return 0;
    if ((uint64_t)a.n_groups * R >= (1ull << 31) * (uint64_t)kW) return 0;   // grid of the codes-only decode
    return (int)R;
}

cudaError_t launch_compress_fast(int R, const CodecArgs& a, uint32_t* flags, cudaStream_t st, unsigned long long* pack_status) {
    return a.dtype == DT_F16 ? compress_fast_t<__half>(R, a, flags, st, pack_status)
                             : compress_fast_t<__nv_bfloat16>(R, a, flags, st, pack_status);
}

cudaError_t launch_decompress_fast(int R, const CodecArgs& a, const DecodeScratch& scratch, cudaStream_t st) {
    return a.dtype == DT_F16 ? decompress_fast_t<__half>(R, a, scratch, st)
                             : decompress_fast_t<__nv_bfloat16>(R, a, scratch, st);
}

}  // namespace speckv

