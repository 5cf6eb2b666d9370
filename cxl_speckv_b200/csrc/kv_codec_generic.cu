// kv_codec_generic.cu -- KV block codec, generic path (any group size / alignment).
//
// One CTA owns one group at a time and walks it in tiles, carrying the encoder
// state (last code, last delta, last natural change, last run head, pairs
// emitted) from tile to tile, so delta and RLE run over the whole flat group
// exactly as the reference does (src/fpga_engine/cache_engine.cpp:198-239).
// Used for odd group sizes, unaligned buffers and fp32 input; the tuned
// kernels for the common geometries live in kv_codec_fast.cu.
//
// Reference functions replaced:
//   compress   = compute_scale_factor + quantize_to_int8 + delta_encode +
//                run_length_encode                     cache_engine.cpp:40-82,172-239
//   decompress = run_length_decode + delta_decode + dequantize_from_int8
//                                                      cache_engine.cpp:84-116,241-284
#include <algorithm>

#include "codec_math.cuh"
#include "kv_codec.h"
#include "device_ctx.h"

namespace speckv {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kEPT = 16;                     // elements per thread per tile (compress)
constexpr int kTile = kThreads * kEPT;       // 4096 elements
constexpr int kPPT = 8;                      // pairs per thread per chunk (decompress)
constexpr int kChunk = kThreads * kPPT;      // 2048 pairs

__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// Groups a CTA works on: g = blockIdx.x + t * gridDim.x, t = 0, 1, ...  With a flag array (second
// pass after the tuned kernels, where almost no group is flagged) the CTA fetches the flags of its
// next 256 groups with one batch of loads, keeps them as 8 ballot words in shared memory and visits
// only the set bits: skipping costs one load latency per 256 groups instead of one per group, and
// flagged groups stay spread over all CTAs.  next() must be called by all threads of the CTA; the
// result is uniform.
struct GroupIter {
    const uint32_t* flags;
    uint32_t n, t0, word, mask;   // t0 = first local index of the NEXT chunk
    uint32_t* smask;              // kWarps words of shared memory
    __device__ GroupIter(const uint32_t* f, uint32_t n_groups, uint32_t* sm)
        : flags(f), n(n_groups), t0(0), word(kWarps), mask(0), smask(sm) {}
    __device__ bool next(uint32_t& g) {
        if (!flags) {   // 64-bit index: n_groups may be close to 2^32, where blockIdx.x + t0 * gridDim.x wraps
            const uint64_t gi = (uint64_t)blockIdx.x + (uint64_t)t0 * gridDim.x;
            ++t0;
            g = (uint32_t)gi;
            return gi < n;
        }
        for (;;) {
            if (mask) {
                const uint32_t j = (uint32_t)__ffs((int)mask) - 1u;
                mask &= mask - 1u;
                g = (uint32_t)((uint64_t)blockIdx.x + (uint64_t)(t0 - kThreads + (word - 1u) * 32u + j) * gridDim.x);   // < n: its flag was read
                return true;
            }
            if (word == kWarps) {   // flags of the CTA's next kThreads groups
                if ((uint64_t)blockIdx.x + (uint64_t)t0 * gridDim.x >= n) return false;
                __syncthreads();    // everybody is done with the previous chunk's words
                const uint64_t i = (uint64_t)blockIdx.x + (uint64_t)(t0 + threadIdx.x) * gridDim.x;
                const unsigned b = __ballot_sync(0xffffffffu, i < n && flags[i] == 1u);   // 2 = the run-expansion path's
                if ((threadIdx.x & 31) == 0) smask[threadIdx.x >> 5] = b;
                __syncthreads();
                t0 += kThreads;
                word = 0;
            }
            mask = smask[word++];
        }
    }
};

// exclusive block scans; `wbuf` holds one int per warp.  Two __syncthreads each.
__device__ __forceinline__ int block_excl_sum(int v, int& total, int* wbuf) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wbuf[wid] = inc;
    __syncthreads();
    int before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        int x = wbuf[w];
        if (w < wid) before += x;
        tot += x;
    }
    __syncthreads();
    total = tot;
    return before + inc - v;
}

__device__ __forceinline__ int block_excl_max(int v, int& total, int* wbuf) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc = max(inc, t);
    }
    int excl = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) excl = -1;
    if (lane == 31) wbuf[wid] = inc;
    __syncthreads();
    int before = -1, tot = -1;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        int x = wbuf[w];
        if (w < wid) before = max(before, x);
        tot = max(tot, x);
    }
    __syncthreads();
    total = tot;
    return max(before, excl);
}

__device__ __forceinline__ float block_max_f(float v, float* wbuf) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (lane == 0) wbuf[wid] = v;
    __syncthreads();
    float m = wbuf[0];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) m = fmaxf(m, wbuf[w]);
    __syncthreads();
    return m;
}

// max |x| over one group, coalesced 128-bit loads when the group is 16 B aligned
template <typename T>
__device__ __forceinline__ float group_absmax(const T* __restrict__ gin, uint32_t G, bool vec_ok, float* wbuf) {
    constexpr int VN = 16 / sizeof(T);
    float m = 0.0f;
    uint32_t done = 0;
    if (vec_ok) {
        const uint32_t nvec = G / VN;
        const uint4* p = reinterpret_cast<const uint4*>(gin);
        for (uint32_t v = threadIdx.x; v < nvec; v += kThreads) {
            uint4 w = ldg_stream(p + v);
            const T* e = reinterpret_cast<const T*>(&w);
#pragma unroll
            for (int j = 0; j < VN; ++j) m = absmax_step(m, widen<T>(e[j]));
        }
        done = nvec * VN;
    }
    for (uint32_t i = done + threadIdx.x; i < G; i += kThreads) m = absmax_step(m, widen<T>(gin[i]));
    return block_max_f(m, wbuf);
}

template <typename T>
__device__ __forceinline__ void load_elems(const T* __restrict__ gin, uint32_t start, uint32_t G, bool vec_ok,
                                           float (&x)[kEPT]) {
    if (vec_ok && start + kEPT <= G) {
        constexpr int NV = kEPT * sizeof(T) / 16;
        uint4 v[NV];
        const uint4* p = reinterpret_cast<const uint4*>(gin + start);
#pragma unroll
        for (int i = 0; i < NV; ++i) v[i] = __ldg(p + i);
        const T* e = reinterpret_cast<const T*>(v);
#pragma unroll
        for (int j = 0; j < kEPT; ++j) x[j] = widen<T>(e[j]);
    } else {
#pragma unroll
        for (int j = 0; j < kEPT; ++j) x[j] = (start + j < G) ? widen<T>(gin[start + j]) : 0.0f;
    }
}

// ---------------------------------------------------------------------------------
// compress, scheme INT8_DELTA_RLE
// ---------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
compress_rle_generic_kernel(const __grid_constant__ CodecArgs a, const uint32_t* __restrict__ only_flagged) {
    __shared__ __align__(16) uint16_t stage[kTile + 16];
    __shared__ int wbuf[kWarps];
    __shared__ float fbuf[kWarps];
    __shared__ uint32_t sh_q[kThreads], sh_d[kThreads];
    __shared__ uint32_t carry_sm[3];
    const int tid = threadIdx.x;

    __shared__ uint32_t smask[kWarps];
    const uint32_t G = a.group_elems;
    GroupIter it(only_flagged, a.n_groups, smask);
    for (uint32_t g; it.next(g);) {
        const T* gin = a.elem_block(static_cast<const T*>(a.in), g, G);
        uint8_t* gout = a.block_payload(g);   // packed emission: the slot reserved by the tuned kernel
        const bool vec_ok = (reinterpret_cast<uintptr_t>(gin) & 15) == 0;
        const uint32_t n = a.group_length(g, G);

        // second pass behind the tuned kernel: that kernel already took the group max and left its bits in
        // comp_bytes[g] (overwritten with the size below), so the input is read once here, not twice
        const float m = only_flagged ? __uint_as_float(a.comp_bytes[g]) : group_absmax<T>(gin, n, vec_ok, fbuf);
        const float s = scale_for(m, scheme_max_scale(a.scheme));
        const bool fast = fast_quant_ok<T>(m);
        float r = 0.0f, rl = 0.0f;
        if (fast) recip_hi_lo(s, r, rl);

        uint32_t carry_q = 0, carry_d = 0;
        int carry_p0 = 0, carry_lh = 0, carry_nh = 0, stage_base = 0;

        for (uint32_t tile = 0; tile < n; tile += kTile) {
            const uint32_t start = tile + tid * kEPT;
            const int cnt = start < n ? min((uint32_t)kEPT, n - start) : 0;
            float x[kEPT];
            load_elems<T>(gin, start, n, vec_ok, x);
            uint32_t q[kEPT];
            if (fast) {
#pragma unroll
                for (int j = 0; j < kEPT; ++j) q[j] = quantize_fast(x[j], r, rl);
            } else {
#pragma unroll
                for (int j = 0; j < kEPT; ++j) q[j] = quantize_exact(x[j], s);
            }
            if (cnt > 0) sh_q[tid] = q[cnt - 1];
            __syncthreads();
            const uint32_t prev_q = tid == 0 ? carry_q : sh_q[tid - 1];
            uint32_t d[kEPT];
#pragma unroll
            for (int j = 0; j < kEPT; ++j) d[j] = (q[j] - (j ? q[j - 1] : prev_q)) & 0xffu;
            if (cnt > 0) sh_d[tid] = d[cnt - 1];
            __syncthreads();
            const uint32_t prev_d = tid == 0 ? carry_d : sh_d[tid - 1];

            // natural run boundaries: delta differs from its predecessor (position 0 always)
            uint32_t chg = 0;
#pragma unroll
            for (int j = 0; j < kEPT; ++j) {
                const bool c = (start + j == 0) || (d[j] != (j ? d[j - 1] : prev_d));
                if (j < cnt && c) chg |= 1u << j;
            }
            int tot_lc;
            const int lc = chg ? (int)start + (31 - __clz(chg)) : -1;
            const int p0_in = max(carry_p0, block_excl_max(lc, tot_lc, wbuf));

            // run heads = natural boundaries + a forced cut every 255 elements (count < 255, :223)
            const int lh_in = start > 0 ? p0_in + 255 * (((int)start - 1 - p0_in) / 255) : 0;
            int lh = lh_in;
            uint32_t heads = 0;
#pragma unroll
            for (int j = 0; j < kEPT; ++j) {
                const int pos = (int)start + j;
                if (j < cnt && (((chg >> j) & 1u) || pos - lh == 255)) {
                    heads |= 1u << j;
                    lh = pos;
                }
            }
            int tot_h;
            int nh = carry_nh + block_excl_sum(__popc(heads), tot_h, wbuf);

            // a head at pos closes the previous run: pair (delta[pos-1], pos - head_of_that_run)
            int lh2 = lh_in;
            uint32_t dprev = prev_d;
#pragma unroll
            for (int j = 0; j < kEPT; ++j) {
                if ((heads >> j) & 1u) {
                    const int pos = (int)start + j;
                    if (pos > 0) stage[(nh - 1) - stage_base] = (uint16_t)(dprev | ((uint32_t)(pos - lh2) << 8));
                    ++nh;
                    lh2 = pos;
                }
                dprev = d[j];
            }
            const uint32_t last_valid = min(n, tile + kTile) - 1;
            if (cnt > 0 && start + cnt - 1 == last_valid) {
                carry_sm[0] = q[cnt - 1];
                carry_sm[1] = d[cnt - 1];
                carry_sm[2] = (uint32_t)lh;
            }
            __syncthreads();
            carry_q = carry_sm[0];
            carry_d = carry_sm[1];
            carry_lh = (int)carry_sm[2];
            carry_p0 = max(carry_p0, tot_lc);
            carry_nh += tot_h;

            // stream out the completed pairs in whole 16-byte vectors, keep the tail
            const int avail = (carry_nh - 1) - stage_base;
            const int nvec = avail >> 3;
            uint4* dst = reinterpret_cast<uint4*>(gout + (size_t)stage_base * 2);
            const uint4* src = reinterpret_cast<const uint4*>(stage);
            for (int v = tid; v < nvec; v += kThreads) dst[v] = src[v];
            const int rem = avail - (nvec << 3);
            const uint16_t keep = tid < rem ? stage[(nvec << 3) + tid] : (uint16_t)0;
            __syncthreads();
            if (tid < rem) stage[tid] = keep;
            stage_base += nvec << 3;
        }

        __syncthreads();
        if (n > 0) {
            // the run still open at the end of the group (:235-236)
            const int rem = (carry_nh - 1) - stage_base;  // pairs waiting in the stage, < 8
            if (tid == 0) stage[rem] = (uint16_t)(carry_d | ((uint32_t)((int)n - carry_lh) << 8));
            if (tid > rem && tid < 8) stage[tid] = 0;
            __syncthreads();
            if (tid == 0) *reinterpret_cast<uint4*>(gout + (size_t)stage_base * 2) = *reinterpret_cast<const uint4*>(stage);
        }
        if (tid == 0) {
            a.scales[g] = s;
            a.comp_bytes[g] = 2u * (uint32_t)carry_nh;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------
// decompress, run expansion: the groups the tuned kernel flagged 2 (payloads whose runs outgrow its in-place
// staging: constant stretches, zero tails, smooth data -- the regime where the codec actually compresses)
// ---------------------------------------------------------------------------------
// Output-stationary, one warp per OUTPUT region of 2048 elements, warps of the whole grid striding over
// (flagged group, region) items, so a single flagged group still spreads over many warps.  The tuned kernel left,
// per pairs-region, the number of elements and the code before it (DecodeScratch::prefix): a warp finds the
// pairs-region its outputs start in, scans pairs from there (256 per step, counts and code advance by dp4a + one
// warp scan), and records what its 2048 outputs need: one bit per output where a pair starts, the pairs' values in
// table order, the code in front of the region.  Expansion then is the tuned kernel's arithmetic -- 8 deltas per
// lane, running byte sums by dp4a, one warp scan, dequantise, one 16-byte store per lane -- after a gather: the
// lane's 8 deltas are table bytes picked by a byte permute whose selector comes from a 256-entry table indexed by
// the lane's 8 head bits.  Cost per element does not depend on the run lengths.  Counts are >= 1 here (payloads
// with empty pairs keep to the generic kernel) and the decoded length is <= G.
template <typename T> __device__ __forceinline__ uint32_t pack2_bits(float a, float b) { return 0u; }
template <> __device__ __forceinline__ uint32_t pack2_bits<__half>(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
template <> __device__ __forceinline__ uint32_t pack2_bits<__nv_bfloat16>(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

constexpr int kRunsTable = 2048 + 256 + 16;       // values of the pairs that can touch one output region (+ first partial step)
struct RunsSmem {
    uint32_t lut[256];                            // head bits of 8 outputs -> the two byte-permute selectors
    uint32_t bitmap[kWarps][64];                  // bit i: output i of the region starts a pair
    uint32_t wprefix[kWarps][64];                 // pairs started before bitmap word w
    uint32_t table[kWarps][kRunsTable / 4];       // pair values, one byte each
};

template <typename T>
__device__ __forceinline__ void decode_runs_region(RunsSmem& rs, int wid, int lane, const uint8_t* __restrict__ gp,
                                                   uint32_t npairs, float s, const uint2* __restrict__ pre, uint32_t R,
                                                   uint32_t o, T* __restrict__ gout) {
    constexpr unsigned kAll = 0xffffffffu;
    const uint32_t O0 = o * 2048u;
    const uint32_t e_total = __ldg(pre + R).x;
    if (O0 >= e_total) return;
    const uint32_t n_out = min(2048u, e_total - O0), Oend = O0 + n_out;
    uint32_t* bm = rs.bitmap[wid];
    uint32_t* wp = rs.wprefix[wid];
    uint32_t* tb = rs.table[wid];
    bm[lane] = 0u;
    bm[lane + 32] = 0u;
    // pairs-region the outputs start in = the number of regions that END at or before O0 (empty ones included);
    // every lane holds up to four of the (elements, code) prefixes, the one of that region comes by shuffle
    uint2 mine[4];
    uint32_t cnt = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t r = (uint32_t)lane + 32u * i;
        mine[i] = r < R ? __ldg(pre + r + 1) : make_uint2(0xffffffffu, 0u);
        cnt += (r < R && mine[i].x <= O0) ? 1u : 0u;
    }
    const uint32_t r0 = __reduce_add_sync(kAll, cnt);
    uint32_t ecur = 0, qcur = 0;                  // before pairs-region 0: nothing, code 0
    if (r0 > 0) {
        const uint32_t src = (r0 - 1u) & 31u, slot = (r0 - 1u) >> 5;
        uint32_t ex = 0, qx = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t a = __shfl_sync(kAll, mine[i].x, src), b = __shfl_sync(kAll, mine[i].y, src);
            if (slot == (uint32_t)i) {
                ex = a;
                qx = b;
            }
        }
        ecur = ex;
        qcur = qx & 0xffu;
    }
    __syncwarp();
    // ---- scan: head bits, value table, code in front of the region ----
    uint32_t tbase = 0xffffffffu;                 // first pair of the first step that touches the region
    uint32_t found = 0;                           // this lane saw the pair that covers O0: (table index << 8) | code at O0 - 1
    bool have = false;
    for (uint32_t pk = r0 * 2048u; pk < npairs && ecur < Oend; pk += 256u) {
        const uint32_t pb = pk + 8u * lane;
        const int nv = pb < npairs ? (int)min(8u, npairs - pb) : 0;
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
        if (nv > 0) w = ldg_stream(reinterpret_cast<const uint4*>(gp + (size_t)pb * 2));   // slots are 16-byte aligned and so is pb * 2
        if (nv < 8) {
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
        const uint32_t cl = __dp4a(cb, 0x01010101u, __dp4a(ca, 0x01010101u, 0u));
        const uint32_t sl = __dp4a(vb, cb, __dp4a(va, ca, 0u)) & 0xffu;
        const uint32_t own = cl | (sl << 24);
        uint32_t inc = own;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(kAll, inc, d);
            if (lane >= d) inc += t;
        }
        const uint32_t tot = __shfl_sync(kAll, inc, 31);
        const uint32_t step_end = ecur + (tot & 0xffffffu);
        if (step_end > O0) {
            if (tbase == 0xffffffffu) tbase = pk;
            const uint32_t ti = pk - tbase + 8u * lane;
            if (ti + 8u <= (uint32_t)kRunsTable) *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(tb) + ti) = make_uint2(va, vb);
            uint32_t p = ecur + ((inc - own) & 0xffffffu);
            uint32_t q = qcur + ((inc - own) >> 24);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t v = (j < 4 ? va >> (8 * j) : vb >> (8 * (j - 4))) & 0xffu;
                const uint32_t c = (j < 4 ? ca >> (8 * j) : cb >> (8 * (j - 4))) & 0xffu;
                if (c != 0u && p < Oend && p + c > O0) {
                    const uint32_t pos = max(p, O0) - O0;
                    atomicOr(&bm[pos >> 5], 1u << (pos & 31u));
                    if (p <= O0) {
                        have = true;
                        found = ((ti + (uint32_t)j) << 8) | ((q + v * (O0 - p)) & 0xffu);
                    }
                }
                p += c;
                q += v * c;
            }
        }
        ecur = step_end;
        qcur = (qcur + (tot >> 24)) & 0xffu;
    }
    const unsigned who = __ballot_sync(kAll, have);
    found = __shfl_sync(kAll, found, who ? __ffs((int)who) - 1 : 0);
    const uint32_t first_ti = found >> 8;
    uint32_t qrun = found & 0xffu;                // code of output O0 - 1
    __syncwarp();
    // heads before every bitmap word (one scan for the whole region; the steps below then need none for the ranks)
    {
        const uint32_t w0 = bm[2 * lane], w1 = bm[2 * lane + 1];
        const uint32_t n0 = (uint32_t)__popc(w0), n1 = (uint32_t)__popc(w1);
        uint32_t inc = n0 + n1;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(kAll, inc, d);
            if (lane >= d) inc += t;
        }
        wp[2 * lane] = inc - n0 - n1;
        wp[2 * lane + 1] = inc - n1;
    }
    __syncwarp();
    // ---- expansion: 256 outputs per step, 8 per lane ----
    for (uint32_t k0 = 0; k0 < n_out; k0 += 256u) {
        const uint32_t wi0 = (k0 >> 5) + (lane >> 2), bsh = 8u * (lane & 3u);
        const uint32_t word = bm[wi0];
        const uint32_t hb = (word >> bsh) & 0xffu;
        const uint32_t before = wp[wi0] + (uint32_t)__popc(word & ((1u << bsh) - 1u));   // heads before the lane's chunk
        // table index of the pair the lane's first byte comes from: the pair running into the chunk, or -- when the
        // chunk's first output starts a pair -- that pair (the selectors count from there)
        const uint32_t a = first_ti + before - 1u + (hb & 1u);
        const uint32_t wi = a >> 2, sh = (a & 3u) * 8u;
        const uint32_t x0 = tb[wi], x1 = tb[wi + 1], x2 = tb[wi + 2];
        const uint32_t t0 = __funnelshift_r(x0, x1, sh), t1 = __funnelshift_r(x1, x2, sh);
        const uint32_t sel = rs.lut[hb];
        const uint32_t d0 = __byte_perm(t0, t1, sel & 0xffffu), d1 = __byte_perm(t0, t1, sel >> 16);
        const uint32_t sl = __dp4a(d1, 0x01010101u, __dp4a(d0, 0x01010101u, 0u));
        uint32_t inc = sl;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(kAll, inc, d);
            if (lane >= d) inc += t;
        }
        const uint32_t qb = qrun + inc - sl;
        const uint32_t q4 = __dp4a(d0, 0x01010101u, qb);
        const uint32_t q8 = __dp4a(d1, 0x01010101u, q4);
        float y[8];
        y[0] = dequantize(__dp4a(d0, 0x00000001u, qb), s);
        y[1] = dequantize(__dp4a(d0, 0x00000101u, qb), s);
        y[2] = dequantize(__dp4a(d0, 0x00010101u, qb), s);
        y[3] = dequantize(q4, s);
        y[4] = dequantize(__dp4a(d1, 0x00000001u, q4), s);
        y[5] = dequantize(__dp4a(d1, 0x00000101u, q4), s);
        y[6] = dequantize(__dp4a(d1, 0x00010101u, q4), s);
        y[7] = dequantize(q8, s);
        const uint32_t e = k0 + 8u * lane;
        if (sizeof(T) == 2 && e + 8u <= n_out) {
            *reinterpret_cast<uint4*>(gout + O0 + e) = make_uint4(pack2_bits<T>(y[0], y[1]), pack2_bits<T>(y[2], y[3]),
                                                                  pack2_bits<T>(y[4], y[5]), pack2_bits<T>(y[6], y[7]));
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (e + j < n_out) gout[O0 + e + j] = narrow<T>(y[j]);
        }
        qrun = (qrun + __shfl_sync(kAll, inc, 31)) & 0xffu;
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------
// decompress, scheme INT8_DELTA_RLE
// ---------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
decompress_rle_generic_kernel(const __grid_constant__ CodecArgs a, const uint32_t* __restrict__ only_flagged, const DecodeScratch runs) {
    const uint32_t G = a.group_elems, n_groups = a.live_groups();
    T* out = static_cast<T*>(a.out);
    // ---- first the groups flagged for run expansion: warps of the whole grid stride over (group, output region) ----
    if (runs.counters) {
        __shared__ RunsSmem rs;
        const uint32_t n_runs = *reinterpret_cast<const volatile uint32_t*>(runs.counters);
        if (n_runs) {
            {   // selectors: output j of a chunk takes table byte popc(heads up to and including j) - (head at 0)
                const uint32_t hb = threadIdx.x;
                uint32_t sel = 0;
                for (int j = 0; j < 8; ++j) {
                    const uint32_t idx = (uint32_t)__popc(hb & ((2u << j) - 1u)) - (hb & 1u);
                    sel |= (idx & 7u) << (4 * j);
                }
                rs.lut[hb] = sel;
            }
            __syncthreads();
            const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
            const uint32_t R = runs.regions;
            const uint64_t n_items = (uint64_t)n_runs * R;
            for (uint64_t it = (uint64_t)blockIdx.x * kWarps + wid; it < n_items; it += (uint64_t)gridDim.x * kWarps) {
                const uint32_t g = __ldg(runs.list + it / R), o = (uint32_t)(it % R);
                const uint32_t gi = a.stored_block(g);
                const uint32_t npairs = min(__ldg(a.comp_bytes + gi) >> 1, R * 2048u);
                decode_runs_region<T>(rs, wid, lane, a.block_payload(gi), npairs, __ldg(a.scales + gi), runs.prefix + (size_t)g * (R + 1),
                                      R, o, a.elem_block(out, g, G));
            }
            // the last CTA to get here clears the list for the next call (every CTA has read the count by then).  Only
            // when there was a list: with n_runs == 0 both counters are zero already, and one atomic per CTA on the same
            // word made the (usual) empty second pass twice as long as it needs to be.
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                if (atomicAdd(runs.counters + 1, 1u) == gridDim.x - 1) {
                    runs.counters[0] = 0u;
                    runs.counters[1] = 0u;
                }
            }
        }
    }
    // Output-stationary expansion: a chunk of 2048 pairs is scanned once (start position and
    // starting code of every pair go to shared memory); then every thread produces 16 consecutive
    // output elements at a time -- binary search for the pair covering its first element, then a
    // walk -- so the cost per element does not depend on the run lengths (a block of zeros is 515
    // pairs of 255 elements each) and the stores are whole 16-byte vectors.
    constexpr int V = 16 / sizeof(T);
    constexpr int kOut = 16;                         // elements per thread per window
    // per pair: x = output position where it starts, y = code before it | value << 8 | count << 16
    __shared__ uint2 s_ent[kChunk + 1];              // (+ end sentinel)
    __shared__ int wbuf[kWarps];
    const int tid = threadIdx.x;

    __shared__ uint32_t smask[kWarps];
    GroupIter it(only_flagged, n_groups, smask);
    for (uint32_t g; it.next(g);) {
        const uint32_t gi = a.stored_block(g);
        const uint8_t* gp = a.block_payload(gi);
        uint32_t npairs = __ldg(a.comp_bytes + gi) >> 1;  // a trailing odd byte is ignored (:245-247)
        npairs = min(npairs, (uint32_t)(a.slot_bytes >> 1));
        const float s = __ldg(a.scales + gi);
        const bool special = scale_is_special(s);
        T* gout = a.elem_block(out, g, G);
        const bool vec_ok = (reinterpret_cast<uintptr_t>(gout) & 15) == 0;
        const bool in_vec_ok = (reinterpret_cast<uintptr_t>(gp) & 15) == 0;

        uint32_t out_pos = 0, acc = 0;
        for (uint32_t c0 = 0; c0 < npairs && out_pos < G; c0 += kChunk) {
            const uint32_t pbase = c0 + tid * kPPT;
            const int np = pbase < npairs ? min((uint32_t)kPPT, npairs - pbase) : 0;
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            if (np == kPPT && in_vec_ok) {
                uint4 t = ldg_stream(reinterpret_cast<const uint4*>(gp + (size_t)pbase * 2));
                w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
            } else {
                const uint16_t* p16 = reinterpret_cast<const uint16_t*>(gp) + pbase;
                for (int k = 0; k < np; ++k) w[k >> 1] |= (uint32_t)p16[k] << (16 * (k & 1));
            }
            uint32_t C = 0, S = 0;
#pragma unroll
            for (int k = 0; k < kPPT; ++k) {
                const uint32_t pr = (w[k >> 1] >> (16 * (k & 1))) & 0xffffu;
                C += pr >> 8;
                S += (pr & 0xffu) * (pr >> 8);
            }
            int totC, totS;
            uint32_t p = out_pos + (uint32_t)block_excl_sum((int)C, totC, wbuf);
            uint32_t qb = acc + (uint32_t)block_excl_sum((int)S, totS, wbuf);
#pragma unroll
            for (int k = 0; k < kPPT; ++k) {
                const uint32_t pr = (w[k >> 1] >> (16 * (k & 1))) & 0xffffu;
                s_ent[tid * kPPT + k] = make_uint2(p, (qb & 0xffu) | (pr << 8));
                p += pr >> 8;
                qb += (pr & 0xffu) * (pr >> 8);
            }
            if (tid == kThreads - 1) s_ent[kChunk] = make_uint2(p, 0u);   // == out_pos + totC
            __syncthreads();
            const uint32_t chunk_end = (uint32_t)min((uint64_t)out_pos + (uint64_t)totC, (uint64_t)G);
            // windows of kThreads * kOut elements aligned to the group start
            for (uint32_t w0 = (out_pos / (kThreads * kOut)) * (kThreads * kOut); w0 < chunk_end; w0 += kThreads * kOut) {
                const uint32_t e0 = w0 + tid * kOut;
                const uint32_t lo = max(e0, out_pos), hi = min(e0 + kOut, chunk_end);
                if (lo >= hi) continue;
                // last pair whose start is <= lo (pairs with count 0 share their start with the next one)
                uint32_t a = 0, b = kChunk;   // invariant: pos[a] <= lo < pos[b]
                while (b - a > 1) {
                    const uint32_t mid = (a + b) >> 1;
                    if (s_ent[mid].x <= lo) a = mid; else b = mid;
                }
                uint32_t j = a;
                uint2 en = s_ent[j];          // en.y: code before | value << 8 | count << 16
                T vals[kOut];
#pragma unroll
                for (int i = 0; i < kOut; ++i) {
                    const uint32_t e = e0 + i;
                    if (e >= lo && e < hi) {
                        while (e >= en.x + (en.y >> 16)) en = s_ent[++j];   // next pair (skips empty ones)
                        const uint32_t code = en.y + ((en.y >> 8) & 0xffu) * (e - en.x + 1u);
                        vals[i] = special ? narrow_special<T>(dequantize_special(code & 0xffu, s)) : narrow<T>(dequantize(code, s));
                    } else {
                        vals[i] = narrow<T>(0.0f);
                    }
                }
                if (vec_ok && lo == e0 && hi == e0 + kOut) {
                    uint4* dst = reinterpret_cast<uint4*>(gout + e0);
                    const uint4* src = reinterpret_cast<const uint4*>(vals);
#pragma unroll
                    for (int v = 0; v < kOut / V; ++v) dst[v] = src[v];
                } else {
#pragma unroll
                    for (int i = 0; i < kOut; ++i)
                        if (e0 + i >= lo && e0 + i < hi) gout[e0 + i] = vals[i];
                }
            }
            __syncthreads();   // the chunk tables are rewritten by the next chunk
            out_pos = chunk_end;
            acc = (acc + (uint32_t)totS) & 0xffu;
        }
        if (tid == 0 && a.out_elems) a.out_elems[g] = out_pos;
    }
}

// ---------------------------------------------------------------------------------
// scheme INT8: codes only (quantize_to_int8 / dequantize_from_int8)
// ---------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
compress_int8_generic_kernel(const __grid_constant__ CodecArgs a, const uint32_t* __restrict__ only_flagged) {
    __shared__ float fbuf[kWarps];
    __shared__ uint32_t smask[kWarps];
    const int tid = threadIdx.x;
    const uint32_t G = a.group_elems;
    GroupIter it(only_flagged, a.n_groups, smask);
    for (uint32_t g; it.next(g);) {
        const T* gin = a.elem_block(static_cast<const T*>(a.in), g, G);
        uint8_t* gout = static_cast<uint8_t*>(a.payload) + (size_t)g * a.slot_bytes;   // no packed emission with codes only
        const bool vec_ok = (reinterpret_cast<uintptr_t>(gin) & 15) == 0;
        const uint32_t n = a.group_length(g, G);
        // behind the tuned kernel the group max is already known (left in comp_bytes[g])
        const float m = only_flagged ? __uint_as_float(a.comp_bytes[g]) : group_absmax<T>(gin, n, vec_ok, fbuf);
        const float s = scale_for(m, scheme_max_scale(a.scheme));
        const bool fast = fast_quant_ok<T>(m);
        float r = 0.0f, rl = 0.0f;
        if (fast) recip_hi_lo(s, r, rl);
        for (uint32_t tile = 0; tile < n; tile += kTile) {
            const uint32_t start = tile + tid * kEPT;
            float x[kEPT];
            load_elems<T>(gin, start, n, vec_ok, x);
            uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int j = 0; j < kEPT; ++j) {
                const uint32_t q = fast ? quantize_fast(x[j], r, rl) : quantize_exact(x[j], s);
                w[j >> 2] |= q << (8 * (j & 3));
            }
            if (start + kEPT <= n) {
                *reinterpret_cast<uint4*>(gout + start) = make_uint4(w[0], w[1], w[2], w[3]);
            } else {
                for (uint32_t j = 0; start + j < n && j < kEPT; ++j) gout[start + j] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
            }
        }
        if (tid == 0) {
            a.scales[g] = s;
            a.comp_bytes[g] = n;
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
decompress_int8_generic_kernel(const __grid_constant__ CodecArgs a, const uint32_t* __restrict__ only_flagged) {
    __shared__ uint32_t smask[kWarps];
    const int tid = threadIdx.x;
    const uint32_t G = a.group_elems;
    GroupIter it(only_flagged, a.live_groups(), smask);
    for (uint32_t g; it.next(g);) {
        const uint32_t gi = a.stored_block(g);
        const uint8_t* gp = a.block_payload(gi);
        const uint32_t n = min(min(__ldg(a.comp_bytes + gi), G), (uint32_t)a.slot_bytes);
        const float s = __ldg(a.scales + gi);
        T* gout = a.elem_block(static_cast<T*>(a.out), g, G);
        const bool special = scale_is_special(s);
        for (uint32_t i = tid; i < n; i += kThreads)
            gout[i] = special ? narrow_special<T>(dequantize_special(__ldg(gp + i), s)) : narrow<T>(dequantize(__ldg(gp + i), s));
        if (tid == 0 && a.out_elems) a.out_elems[g] = n;
    }
}

// scheme FP16: raw 16-bit passthrough of fp16 / bf16 groups
// raw copy of whole groups into their slots (and the metadata), 16 bytes per thread and step when both sides allow
__global__ void __launch_bounds__(kThreads)
passthrough_in_kernel(const __grid_constant__ CodecArgs a) {
    const uint16_t* in = static_cast<const uint16_t*>(a.in);
    uint8_t* payload = static_cast<uint8_t*>(a.payload);
    const size_t slot_bytes = a.slot_bytes;
    const uint32_t G = a.group_elems, n_groups = a.n_groups;
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(payload) | slot_bytes) & 15) == 0 && G % 8 == 0;
    const uint64_t vec_per_group = G / 8;
    if (vec_ok) {
        const uint64_t total = (uint64_t)n_groups * vec_per_group;
        for (uint64_t v = (uint64_t)blockIdx.x * kThreads + threadIdx.x; v < total; v += (uint64_t)gridDim.x * kThreads) {
            const uint64_t g = v / vec_per_group, k = v - g * vec_per_group;
            reinterpret_cast<uint4*>(payload + g * slot_bytes)[k] = ldg_stream(reinterpret_cast<const uint4*>(in) + v);
        }
    } else {
        const uint64_t total = (uint64_t)n_groups * G;
        for (uint64_t e = (uint64_t)blockIdx.x * kThreads + threadIdx.x; e < total; e += (uint64_t)gridDim.x * kThreads) {
            const uint64_t g = e / G, k = e - g * G;
            reinterpret_cast<uint16_t*>(payload + g * slot_bytes)[k] = in[e];
        }
    }
    for (uint32_t g = blockIdx.x * kThreads + threadIdx.x; g < n_groups; g += gridDim.x * kThreads) {
        a.scales[g] = 1.0f;
        a.comp_bytes[g] = G * 2u;
    }
}

__global__ void __launch_bounds__(kThreads)
passthrough_out_kernel(const __grid_constant__ CodecArgs a) {
    const uint32_t G = a.group_elems, n_groups = a.live_groups();
    uint16_t* out = static_cast<uint16_t*>(a.out);
    for (uint32_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const uint32_t gi = a.stored_block(g);
        const uint16_t* gp = reinterpret_cast<const uint16_t*>(a.block_payload(gi));
        const uint32_t n = min(min(__ldg(a.comp_bytes + gi) >> 1, G), (uint32_t)(a.slot_bytes >> 1));
        for (uint32_t i = threadIdx.x; i < n; i += kThreads) out[(size_t)g * G + i] = __ldg(gp + i);
        if (threadIdx.x == 0 && a.out_elems) a.out_elems[g] = n;
    }
}

#ifndef SPECKV_SECOND_PASS_PER_SM
#define SPECKV_SECOND_PASS_PER_SM 3
#endif
constexpr int kSecondPassPerSm = SPECKV_SECOND_PASS_PER_SM;
inline int grid_for(uint32_t n_groups, int sm_count, int per_sm) {
    const long long cap = (long long)sm_count * per_sm;
    return (int)((long long)n_groups < cap ? (n_groups ? n_groups : 1) : cap);
}

}  // namespace

template <typename T>
static cudaError_t launch_compress_t(const CodecArgs& a, cudaStream_t st, const uint32_t* only_flagged) {
    // as the second pass behind a tuned kernel almost nothing is flagged: a smaller grid (its launch and drain are
    // what an empty pass costs) still spreads the few flagged groups over every SM
    const int grid = grid_for(a.n_groups, current_sm_count(), only_flagged ? kSecondPassPerSm : 8);
    if (scheme_is_rle(a.scheme)) compress_rle_generic_kernel<T><<<grid, kThreads, 0, st>>>(a, only_flagged);
    else compress_int8_generic_kernel<T><<<grid, kThreads, 0, st>>>(a, only_flagged);
    count_launch();
    return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_decompress_t(const CodecArgs& a, cudaStream_t st, const uint32_t* only_flagged, const DecodeScratch* runs) {
    const int sm_count = current_sm_count();
    int grid = grid_for(a.n_groups, sm_count, only_flagged ? kSecondPassPerSm : 8);
    if (runs) {   // a few flagged groups still spread over the device: one warp per output region, up to 2 CTAs per SM
        const long long want = ((long long)a.n_groups * runs->regions + kWarps - 1) / kWarps;
        const long long cap = (long long)sm_count * 2;
        grid = (int)std::max<long long>(grid, std::min(want, cap));
    }
    if (scheme_is_rle(a.scheme)) decompress_rle_generic_kernel<T><<<grid, kThreads, 0, st>>>(a, only_flagged, runs ? *runs : DecodeScratch{});
    else decompress_int8_generic_kernel<T><<<grid, kThreads, 0, st>>>(a, only_flagged);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_compress_generic(const CodecArgs& a, cudaStream_t st, const uint32_t* only_flagged) {
    if (a.n_groups == 0) return cudaSuccess;
    if (a.scheme == 0) {
        if (a.elem_index) return cudaErrorInvalidValue;   // the raw passthrough has no gather form
        passthrough_in_kernel<<<current_sm_count() * 8, kThreads, 0, st>>>(a);
        count_launch();
        return cudaGetLastError();
    }
    switch (a.dtype) {
        case DT_F16: return launch_compress_t<__half>(a, st, only_flagged);
        case DT_BF16: return launch_compress_t<__nv_bfloat16>(a, st, only_flagged);
        default: return launch_compress_t<float>(a, st, only_flagged);
    }
}

cudaError_t launch_decompress_generic(const CodecArgs& a, cudaStream_t st, const uint32_t* only_flagged, const DecodeScratch* runs) {
    if (a.n_groups == 0) return cudaSuccess;
    if (a.scheme == 0) {
        if (a.elem_index) return cudaErrorInvalidValue;
        passthrough_out_kernel<<<grid_for(a.n_groups, current_sm_count(), 8), kThreads, 0, st>>>(a);
        count_launch();
        return cudaGetLastError();
    }
    switch (a.dtype) {
        case DT_F16: return launch_decompress_t<__half>(a, st, only_flagged, runs);
        case DT_BF16: return launch_decompress_t<__nv_bfloat16>(a, st, only_flagged, runs);
        default: return launch_decompress_t<float>(a, st, only_flagged, runs);
    }
}

}  // namespace speckv
