// prefetch_score.cu -- batched speculative-prefetch scoring, residency filter and request emission.
//
// Replaces LSTMPredictor::predict_top_k (src/prefetcher/lstm_predictor.cpp:40-94) and
// SpeculativePrefetcher::prefetch (src/prefetcher/speculative_prefetcher.cpp:25-82) for a whole
// batch of sequences per call (the reference scores one sequence per call on the CPU: 17.8 ms
// each, SURVEY.md section 6).
//
// What the reference's "LSTM" actually computes (and what is reproduced, step for step):
//   per token t of the 16-token window, per layer (the SAME embedded input and state both times,
//   weights ignored, lstm_predictor.cpp:116-147):
//       g = sum_{j<64} emb[tok][j] * 0.1f        sequential fp32 (mul, then add)      :138-140
//       c = 0.5f*c + 0.5f*tanh(g);  h = 0.5f*tanh(c)                                  :143-145
//   so all 128 hidden units carry the same value h.
//   logit_v = sum_{j<128} h * W[v][j]            sequential fp32 (mul, then add)      :166-173
//   p = softmax(logits) (max-subtracted), top-k by p                                  :176-188,:72-92
//   request i: va = (req << 32) | (layer << 16) | (i + 1)         speculative_prefetcher.cpp:153-160
//   skipped when the page of va is in L1 or L2 (:51-54), else a PrefetchRequest is queued (:57-66)
//
// Three launches, no logits in memory (the first version wrote batch x vocab logits and read them
// back: 32.8 MB next to the 16.4 MB of W_out):
//   hidden_warp_kernel    one warp per sequence: gather the window's embedding rows, 16 x 2 cell updates
//   score_partial_kernel  persistent CTAs walk the vocabulary in tiles of W_out rows staged with cp.async
//                         (double-buffered).  A thread owns S sequences and a few rows of every tile and
//                         keeps, per sequence, the running max, the running sum of exp (online softmax)
//                         and its best K (value, id) in registers.  The logit keeps the reference's
//                         sequential j order; the product of a sequence pair is one packed FMUL2, the
//                         add stays scalar (ptxas would contract a packed mul + packed add into FFMA2,
//                         profiles/micro/f32x2_probe.cu).  The threads of a CTA merge through shared memory:
//                         one partial (max, sum, best K) per CTA and sequence.
//   score_merge_kernel    one warp per sequence merges the CTA partials (sum rescaled in fp64), evaluates the k
//                         confidences, probes the page table for residency, and the last CTA to finish compacts the
//                         surviving PrefetchRequest records in sequence order behind a header that holds their count.
// tanh and the k reported exp values are evaluated in fp64 and rounded once to fp32 (glibc's float versions are
// within 1 ulp of that); parity is "same top-k ids, confidences within 1e-7", not bitwise (SURVEY.md section 8a A11).
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "../../include/speckv_ext.h"
#include "codec_math.cuh"
#include "device_ctx.h"
#include "page_lookup.h"

namespace speckv {

namespace {

struct Predictor {
    float* d_emb = nullptr;
    float* d_wout = nullptr;
    float* d_rowsum = nullptr;   // sum_j W[v][j] (fp64 sum rounded once), the rank-one form of the logits
    uint32_t* d_cand = nullptr;  // the 16 first rows by (rowsum descending, id) and by (rowsum ascending, id)
    float row_abs_max = 0.0f;    // max_v sum_j |W[v][j]| (rounded up): scales the error bound of the rank-one form
    uint32_t vocab = 0, emb_dim = 0, hidden = 0, layers = 0, hist_len = 0;
    int device = -1;
    size_t smem_optin = 0;       // the device's shared memory per block (opt-in): bounds the tiled kernel's W_out tile
    // device-side prefetcher state (SpeculativePrefetcher's queue and counters, speculative_prefetcher.h:83-94)
    speckv_prefetch_request_t* d_ring = nullptr;   // the 16 most recent requests (issue_dma_prefetch, :162-172)
    unsigned long long* d_total = nullptr;         // requests emitted so far
};
std::mutex g_pred_mu;
Predictor g_pred;

// host-side prefetcher statistics (PrefetchStatistics, speculative_prefetcher.h:59-66)
struct EmitCall {
    cudaEvent_t a = nullptr, b = nullptr;
    bool busy = false;
};
constexpr int kEmitCalls = 32;
EmitCall g_calls[kEmitCalls];
unsigned long long* g_h_counts = nullptr;   // pinned + mapped: the merge kernel reports each call's request count here
unsigned long long* g_d_counts = nullptr;   // device view of g_h_counts
uint64_t g_stat_total = 0, g_stat_mispred = 0;
double g_stat_latency_us = 0.0;

constexpr uint32_t kRing = 16;

// Same recurrence, one WARP per sequence: the lanes first gather the window's embedding rows into shared
// memory (hist_len x nj independent loads in flight instead of one dependent load per addition), then lane 0
// runs the reference's sequential sums over them.
constexpr int kHiddenWarps = 4;
__global__ void __launch_bounds__(kHiddenWarps * 32)
hidden_warp_kernel(const uint32_t* __restrict__ tokens, uint32_t batch, uint32_t hist_len,
                   const float* __restrict__ emb, uint32_t vocab, uint32_t emb_dim, uint32_t hidden, uint32_t layers,
                   float* __restrict__ h_out, unsigned int* __restrict__ ticket) {
    extern __shared__ float se[];   // [kHiddenWarps][hist_len][nj]
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) *ticket = 0u;   // "CTAs done" counter of this call's merge kernel
    const uint32_t b = blockIdx.x * kHiddenWarps + warp;
    if (b >= batch) return;
    const uint32_t nj = emb_dim < hidden ? emb_dim : hidden;   // `j < input_dim && j < hidden_dim`, :138
    float* my = se + (size_t)warp * hist_len * nj;
    for (uint32_t idx = lane; idx < hist_len * nj; idx += 32) {
        const uint32_t t = idx / nj, j = idx - t * nj;
        const uint32_t tok = tokens[(size_t)b * hist_len + t];
        my[idx] = tok < vocab ? __ldg(emb + (size_t)tok * emb_dim + j) : 0.0f;   // out-of-vocabulary ids embed to zeros, :149-160
    }
    __syncwarp();
    // The candidate g_t and tanh(g_t) depend on token t alone: lane t computes them (the reference's sequential sum
    // over j stays sequential inside the lane), 32 tokens at a time.  What is left of the recurrence is the cell
    // update, c = 0.5 c + 0.5 tanh(g_t) once per layer, in token order; the hidden value is only read after the last
    // step (every intermediate h = 0.5 tanh(c) of :145 is overwritten before anything uses it).
    float c = 0.0f;
    for (uint32_t t0 = 0; t0 < hist_len; t0 += 32) {
        const uint32_t t = t0 + lane;
        float tg = 0.0f;
        if (t < hist_len) {
            float g = 0.0f;
            for (uint32_t j = 0; j < nj; ++j) g = __fadd_rn(g, __fmul_rn(my[t * nj + j], 0.1f));
            tg = (float)tanh((double)g);
        }
        const uint32_t nt = min(32u, hist_len - t0);
        for (uint32_t i = 0; i < nt; ++i) {
            const float tgi = __shfl_sync(0xffffffffu, tg, (int)i);
            for (uint32_t l = 0; l < layers; ++l) c = __fadd_rn(__fmul_rn(0.5f, c), __fmul_rn(0.5f, tgi));
        }
    }
    if (lane == 0) h_out[b] = (hist_len && layers) ? __fmul_rn(0.5f, (float)tanh((double)c)) : 0.0f;
}
// very long windows / wide embeddings (the staging above would not fit): one thread per sequence
__global__ void hidden_kernel(const uint32_t* __restrict__ tokens, uint32_t batch, uint32_t hist_len,
                              const float* __restrict__ emb, uint32_t vocab, uint32_t emb_dim, uint32_t hidden,
                              uint32_t layers, float* __restrict__ h_out, unsigned int* __restrict__ ticket) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b == 0) *ticket = 0u;
    if (b >= batch) return;
    float h = 0.0f, c = 0.0f;
    const uint32_t nj = emb_dim < hidden ? emb_dim : hidden;
    for (uint32_t t = 0; t < hist_len; ++t) {
        const uint32_t tok = tokens[(size_t)b * hist_len + t];
        float g = 0.0f;
        if (tok < vocab) {
            const float* e = emb + (size_t)tok * emb_dim;
            for (uint32_t j = 0; j < nj; ++j) g = __fadd_rn(g, __fmul_rn(__ldg(e + j), 0.1f));
        }
        const float tg = (float)tanh((double)g);
        for (uint32_t l = 0; l < layers; ++l) {
            c = __fadd_rn(__fmul_rn(0.5f, c), __fmul_rn(0.5f, tg));
            h = __fmul_rn(0.5f, (float)tanh((double)c));
        }
    }
    h_out[b] = h;
}

constexpr int kMaxK = 16;
constexpr int kScoreThreads = 256;
constexpr int kScoreWarps = kScoreThreads / 32;

// a > b in the order of the reference's sort by confidence (softmax is monotone in the logit); ties -> lower id
__device__ __forceinline__ bool better(float av, uint32_t ai, float bv, uint32_t bi) {
    return av > bv || (av == bv && ai < bi);
}

// sorted insertion into a list of K (best first), fully predicated (the lanes of a warp hold different sequences)
template <int K>
__device__ __forceinline__ void list_insert(float (&bv)[K], uint32_t (&bi)[K], float x, uint32_t id) {
    if (better(x, id, bv[K - 1], bi[K - 1])) {
        bv[K - 1] = x;
        bi[K - 1] = id;
    }
#pragma unroll
    for (int i = K - 1; i > 0; --i) {
        const bool sw = better(bv[i], bi[i], bv[i - 1], bi[i - 1]);
        const float tv = bv[i];
        const uint32_t ti = bi[i];
        bv[i] = sw ? bv[i - 1] : tv;
        bi[i] = sw ? bi[i - 1] : ti;
        bv[i - 1] = sw ? tv : bv[i - 1];
        bi[i - 1] = sw ? ti : bi[i - 1];
    }
}

__device__ __forceinline__ uint32_t smem_u32_of(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Row stride of a staged W_out tile in words: 16 B aligned rows (the float4 reads below) for any hidden, bank-staggered.
__host__ __device__ __forceinline__ uint32_t tile_ld(uint32_t hidden) { return ((hidden + 3u) & ~3u) + 4u; }

// One partial per (CTA, sequence): { max, sum of exp(x - max), K values, K ids } = 2 + 2K words.
// Geometry (host-chosen): seq_lanes lanes of a warp hold different sequence slices (S sequences each), the other
// lane bits and the warp index select a row subset; a tile has nsub * rps rows, nsub = kScoreWarps * 32 / seq_lanes.
template <int K, int S>
__global__ void __launch_bounds__(kScoreThreads, 2)
score_partial_kernel(const float* __restrict__ wout, uint32_t vocab, uint32_t hidden, const float* __restrict__ hvec,
                     uint32_t batch, uint32_t seq_lanes, uint32_t rps, uint32_t n_tiles, float* __restrict__ partials) {
    extern __shared__ __align__(16) float sm[];
    constexpr int PW = 2 + 2 * K;                      // words per partial
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rsub_per_warp = 32u / seq_lanes, nsub = kScoreWarps * rsub_per_warp;
    const uint32_t ssub = lane % seq_lanes, rsub = warp * rsub_per_warp + lane / seq_lanes;
    const uint32_t tile_rows = nsub * rps;
    const uint32_t ld = tile_ld(hidden);
    const uint32_t sb = seq_lanes * S;                 // sequences per CTA (grid.y walks the batch)
    const uint32_t seq0 = blockIdx.y * sb + ssub * S;
    const uint32_t h4 = hidden & ~3u;

    float hs[S], m[S], bv[S][K];
    double se[S];   // sum of exp(x - max): fp64, or the many small terms of a peaked softmax round away against the top one
    uint32_t bi[S][K];
#pragma unroll
    for (int i = 0; i < S; ++i) {
        hs[i] = seq0 + i < batch ? hvec[seq0 + i] : 0.0f;
        m[i] = -FLT_MAX;
        se[i] = 0.0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            bv[i][k] = -FLT_MAX;
            bi[i][k] = 0xffffffffu;
        }
    }
    f32x2_t h2[S / 2];
#pragma unroll
    for (int i = 0; i < S / 2; ++i) h2[i] = pack_f32x2(hs[2 * i], hs[2 * i + 1]);

    const uint32_t buf_words = tile_rows * ld;
    auto load_tile = [&](uint32_t tile, uint32_t buf) {
        const uint32_t v0 = tile * tile_rows;
        const uint32_t rows = min(tile_rows, vocab - v0);
        const uint32_t base = smem_u32_of(sm + (size_t)buf * buf_words);
        if ((hidden & 3u) == 0) {
            const uint32_t vec_per_row = hidden >> 2;
            for (uint32_t i = tid; i < rows * vec_per_row; i += kScoreThreads) {
                const uint32_t r = i / vec_per_row, c = i - r * vec_per_row;
                cp_async16(base + (r * ld + 4u * c) * 4u, wout + (size_t)(v0 + r) * hidden + 4u * c);
            }
        } else {
            for (uint32_t i = tid; i < rows * hidden; i += kScoreThreads) {
                const uint32_t r = i / hidden, c = i - r * hidden;
                cp_async4(base + (r * ld + c) * 4u, wout + (size_t)(v0 + r) * hidden + c);
            }
        }
    };

    uint32_t it = 0;
    if (blockIdx.x < n_tiles) load_tile(blockIdx.x, 0);
    cp_async_commit();
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const uint32_t next = tile + gridDim.x;
        if (next < n_tiles) load_tile(next, (it + 1) & 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const float* wt = sm + (size_t)(it & 1) * buf_words;
        const uint32_t v0 = tile * tile_rows;
        for (uint32_t r = 0; r < rps; ++r) {
            const uint32_t row = rsub * rps + r, v = v0 + row;
            if (v >= vocab) break;
            const float* w = wt + row * ld;
            float acc[S];
#pragma unroll
            for (int i = 0; i < S; ++i) acc[i] = 0.0f;
            for (uint32_t j = 0; j < h4; j += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(w + j);
                const float wj[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const f32x2_t w2 = pack_f32x2(wj[jj], wj[jj]);
#pragma unroll
                    for (int i = 0; i < S / 2; ++i) {
                        float p0, p1;
                        unpack_f32x2(mul_f32x2(h2[i], w2), p0, p1);            // h[j] * w, :170
                        acc[2 * i] = __fadd_rn(acc[2 * i], p0);                // logits[i] += ..., sequential in j
                        acc[2 * i + 1] = __fadd_rn(acc[2 * i + 1], p1);
                    }
                }
            }
            for (uint32_t j = h4; j < hidden; ++j) {
                const float wj = w[j];
#pragma unroll
                for (int i = 0; i < S; ++i) acc[i] = __fadd_rn(acc[i], __fmul_rn(hs[i], wj));
            }
#pragma unroll
            for (int i = 0; i < S; ++i) {
                const float x = acc[i];
                if (x > m[i]) {   // online softmax: rescale the running sum to the new max
                    se[i] *= (double)expf(m[i] - x);
                    m[i] = x;
                }
                se[i] += (double)expf(x - m[i]);
                list_insert<K>(bv[i], bi[i], x, v);
            }
        }
        __syncthreads();   // everybody is done with this buffer before the load after next overwrites it
    }
    cp_async_wait<0>();
    __syncthreads();

    // ---- merge inside the CTA: every thread parks its partials, then one thread per sequence combines the row subsets ----
    float* park = sm;   // [nsub][sb][PW], aliases the tile buffers
#pragma unroll
    for (int i = 0; i < S; ++i) {
        float* p = park + ((size_t)rsub * sb + ssub * S + i) * PW;
        p[0] = m[i];
        p[1] = (float)se[i];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            p[2 + k] = bv[i][k];
            p[2 + K + k] = __uint_as_float(bi[i][k]);
        }
    }
    __syncthreads();
    for (uint32_t s = tid; s < sb; s += kScoreThreads) {
        const uint32_t seq = blockIdx.y * sb + s;
        if (seq >= batch) continue;
        float mm = -FLT_MAX;
        for (uint32_t q = 0; q < nsub; ++q) mm = fmaxf(mm, park[((size_t)q * sb + s) * PW]);
        float lv[K];
        double ss = 0.0;
        uint32_t li[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            lv[k] = -FLT_MAX;
            li[k] = 0xffffffffu;
        }
        for (uint32_t q = 0; q < nsub; ++q) {
            const float* p = park + ((size_t)q * sb + s) * PW;
            ss += (double)p[1] * (double)expf(p[0] - mm);
#pragma unroll
            for (int k = 0; k < K; ++k) list_insert<K>(lv, li, p[2 + k], __float_as_uint(p[2 + K + k]));
        }
        float* o = partials + ((size_t)seq * gridDim.x + blockIdx.x) * PW;
        o[0] = mm;
        o[1] = (float)ss;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            o[2 + k] = lv[k];
            o[2 + K + k] = __uint_as_float(li[k]);
        }
    }
}


// ---------------------------------------------------------------------------------------------------------
// Rank-one scoring.  Every hidden unit carries the same value h (lstm_predictor.cpp:143-145), so the reference's
// logit_v = fl(sum_j fl(h * W[v][j])) is, up to rounding, h * rowsum[v].  The standard bound for a recursive fp32 sum of
// n products gives |logit_v - h * rowsum[v]| <= gamma_n * |h| * sum_j |W[v][j]|; with the rounding of rowsum and of the
// product that is err = (n + 3) u / (1 - n u) * |h| * max_v sum_j |W[v][j]|, u = 2^-24 (+ a denormal allowance).
// The ORDER of the approximate logits does not depend on the sequence at all: it is the order of rowsum (h > 0) or its
// reverse (h < 0), so the 16 best rows of either order are found once, when the weights are loaded.  One CTA per sequence:
//   1. candidates = the first KC rows of the order for sign(h).  If the weakest candidate's approximate logit is more
//      than 2 err below the k-th best, every row outside the list is provably below the true k-th best: the true top-k
//      are among the candidates;
//   2. the candidates are re-scored with the reference's exact sequential sum and ranked by that (value, then lower id);
//   3. the softmax denominator is summed over the approximate logits, then the candidates' approximate terms are
//      replaced by their exact ones: S' = S - sum_c exp(a_c - M) + sum_c exp(x_c - M).  Every remaining term is within a
//      factor e^(+-err) of its exact value, so |S' - S_exact| <= S_nc (e^err - 1), S_nc the sum over the other rows, and
//      a confidence c is off by at most c |dS| / S'.  When that could exceed half the tolerance 1e-7 + 2^-22 c at the
//      largest confidence (a peaked predictor: err grows with |h| max_v sum_j |W[v][j]|), the CTA takes the exact pass
//      below; for near-uniform predictors (srand(1) weights: ~1e-10) the candidate pass stands;
//   4. otherwise (near-ties wider than the list, h = 0, non-finite weights, the bound of 3) the CTA walks the vocabulary
//      with exact logits, online softmax and per-thread best-KC lists.
// ids are therefore the exact method's ids.  Output: one partial per sequence in score_partial_kernel's format,
// consumed by score_merge_kernel with n_partials = 1.
constexpr int kCandMax = 16;

// KC rounds of warp arg-max over the heads of the lanes' sorted lists; lane r ends up with the r-th best
template <int KC>
__device__ __forceinline__ void warp_select(float (&lv)[KC], uint32_t (&li)[KC], uint32_t lane, float& win_v, uint32_t& win_i) {
    win_v = -FLT_MAX;
    win_i = 0xffffffffu;
    for (int r = 0; r < KC; ++r) {
        float best = lv[0];
        uint32_t idx = li[0];
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const uint32_t oi = __shfl_xor_sync(0xffffffffu, idx, o);
            if (better(ob, oi, best, idx)) {
                best = ob;
                idx = oi;
            }
        }
        if (li[0] == idx && idx != 0xffffffffu) {
#pragma unroll
            for (int i = 0; i + 1 < KC; ++i) {
                lv[i] = lv[i + 1];
                li[i] = li[i + 1];
            }
            lv[KC - 1] = -FLT_MAX;
            li[KC - 1] = 0xffffffffu;
        }
        if (lane == (uint32_t)r) {
            win_v = best;
            win_i = idx;
        }
    }
}

template <int KC>
__global__ void __launch_bounds__(kScoreThreads)
score_rank1_kernel(const float* __restrict__ wout, const float* __restrict__ rowsum, const uint32_t* __restrict__ cand,
                   uint32_t vocab, uint32_t hidden, const float* __restrict__ hvec, uint32_t batch, uint32_t k,
                   float row_abs_max, uint32_t force_exact, float* __restrict__ partials) {
    constexpr int PW = 2 + 2 * KC;
    __shared__ float s_m[kScoreWarps], s_s[kScoreWarps];
    __shared__ float s_v[kScoreWarps][KC];
    __shared__ uint32_t s_i[kScoreWarps][KC];
    constexpr int kRowChunk = 256;
    __shared__ float s_rows[KC][kRowChunk + 1];   // (+1: the lanes read different rows at the same column)
    __shared__ bool s_flag;                        // the candidate pass cannot bound the confidences: exact pass
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t seq = blockIdx.x;
    if (seq >= batch) return;
    const float h = hvec[seq];
    const float u = 5.9604644775390625e-08f;   // 2^-24
    const float err = fabsf(h) * row_abs_max * ((float)(hidden + 3) * u / (1.0f - (float)hidden * u)) * 1.0001f +
                      (float)(hidden + 3) * 1.5e-45f;
    float* o = partials + (size_t)seq * PW;
    const uint32_t nc = min((uint32_t)KC, vocab);
    const uint32_t* cl = cand + (h < 0.0f ? kCandMax : 0);

    // the whole CTA takes the same decision (same inputs)
    bool exact = force_exact != 0u;
    float M = 0.0f;
    if (!exact) {
        M = __fmul_rn(h, __ldg(rowsum + cl[0]));
        const float a_k = __fmul_rn(h, __ldg(rowsum + cl[k - 1]));
        const float a_last = __fmul_rn(h, __ldg(rowsum + cl[nc - 1]));
        exact = !(vocab <= (uint32_t)KC || a_last < a_k - 2.0f * err);   // also taken for NaN bounds
    }

    float S = 0.0f, xv = -FLT_MAX;
    uint32_t ci = 0xffffffffu;
    if (!exact) {
        // ---- softmax denominator over the approximate logits: independent terms, four accumulators per thread ----
        float acc4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        for (uint32_t v0 = tid; v0 < vocab; v0 += 4 * kScoreThreads) {
#pragma unroll
            for (uint32_t q = 0; q < 4; ++q) {
                const uint32_t v = v0 + q * kScoreThreads;
                if (v < vocab) acc4[q] += __expf(__fmul_rn(h, __ldg(rowsum + v)) - M);
            }
        }
        float ws = (acc4[0] + acc4[1]) + (acc4[2] + acc4[3]);
        for (int o2 = 16; o2 > 0; o2 >>= 1) ws += __shfl_xor_sync(0xffffffffu, ws, o2);
        if (lane == 0) s_s[warp] = ws;
        // ---- exact re-scoring: the CTA stages the candidates' rows (chunks of kRowChunk columns), lane r of warp 0
        //      runs the reference's sequential sum over row r (lstm_predictor.cpp:166-173) ----
        if (warp == 0 && lane < nc) ci = cl[lane];
        float acc = 0.0f;
        for (uint32_t j0 = 0; j0 < hidden; j0 += kRowChunk) {
            const uint32_t nj = min((uint32_t)kRowChunk, hidden - j0);
            for (uint32_t idx = tid; idx < nc * nj; idx += kScoreThreads) {
                const uint32_t r = idx / nj, j = idx - r * nj;
                s_rows[r][j] = __fmul_rn(h, __ldg(wout + (size_t)cl[r] * hidden + j0 + j));   // h[j] * w, :170
            }
            __syncthreads();
            if (warp == 0 && lane < nc)
                for (uint32_t j = 0; j < nj; ++j) acc = __fadd_rn(acc, s_rows[lane][j]);       // logits[i] += ..., in j order
            __syncthreads();
        }
        // ---- warp 0: swap the candidates' approximate terms for their exact ones and bound what is left ----
        if (warp == 0) {
            if (lane < nc) xv = acc;
            float ss = lane < kScoreWarps ? s_s[lane] : 0.0f;
            float ta = lane < nc ? __expf(__fmul_rn(h, __ldg(rowsum + ci)) - M) : 0.0f;   // the term summed above
            float best = xv;
            for (int o2 = 16; o2 > 0; o2 >>= 1) {
                ss += __shfl_xor_sync(0xffffffffu, ss, o2);
                ta += __shfl_xor_sync(0xffffffffu, ta, o2);
                best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o2));
            }
            // the exact terms against the exact maximum: the best candidate contributes exactly 1, so S >= 1 and no
            // confidence can exceed 1 (a rescale by exp(M - best) rounds either way)
            float tx = lane < nc ? expf(xv - best) : 0.0f;
            for (int o2 = 16; o2 > 0; o2 >>= 1) tx += __shfl_xor_sync(0xffffffffu, tx, o2);
            const float s_nc = fmaxf(ss - ta, 0.0f) * expf(M - best);   // the rows outside the list, still approximate
            S = s_nc + tx;
            M = best;
            // each remaining term is within a factor e^(+-err) of its exact value: |dS| <= s_nc (e^err - 1), which moves
            // a confidence c by at most c |dS| / S; the largest one, 1 / S, decides (the bar 1e-7 + 2^-22 c grows with c).
            // The fp32 sum above adds its own relative error, at most (terms per accumulator + 10 tree levels) u.
            const float c1 = 1.0f / S;
            const float gsum = (float)((vocab + 4 * kScoreThreads - 1) / (4 * kScoreThreads) + 10) * u;
            const float dc = c1 * (s_nc * expm1f(err) / S + gsum);
            if (lane == 0) s_flag = !(dc <= 0.5f * (1e-7f + 2.384185791015625e-07f * c1));   // NaN -> exact pass
        }
        __syncthreads();
        exact = s_flag;
        if (!exact && warp != 0) return;
    }
    if (exact) {
        // ---- exact pass over the vocabulary ----
        float m = -FLT_MAX, bv[KC];
        double se = 0.0;   // fp64 sums (see score_partial_kernel), fp32 exponentials
        uint32_t bi[KC];
#pragma unroll
        for (int i = 0; i < KC; ++i) {
            bv[i] = -FLT_MAX;
            bi[i] = 0xffffffffu;
        }
        for (uint32_t v = tid; v < vocab; v += kScoreThreads) {
            const float* w = wout + (size_t)v * hidden;
            float x = 0.0f;
            for (uint32_t j = 0; j < hidden; ++j) x = __fadd_rn(x, __fmul_rn(h, __ldg(w + j)));
            // (accurate expf: this pass's time goes to the sequential logit sums, the approximate one would save nothing)
            if (x > m) {
                se *= (double)expf(m - x);
                m = x;
            }
            se += (double)expf(x - m);
            if (better(x, v, bv[KC - 1], bi[KC - 1])) list_insert<KC>(bv, bi, x, v);
        }
        float wm = m;
        for (int o2 = 16; o2 > 0; o2 >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o2));
        double ws = se * (double)expf(m - wm);   // a thread without rows has se = 0
        for (int o2 = 16; o2 > 0; o2 >>= 1) ws += __shfl_xor_sync(0xffffffffu, ws, o2);
        float wv;
        uint32_t wi;
        warp_select<KC>(bv, bi, lane, wv, wi);
        if (lane == 0) {
            s_m[warp] = wm;
            s_s[warp] = (float)ws;
        }
        if (lane < KC) {
            s_v[warp][lane] = wv;
            s_i[warp][lane] = wi;
        }
        __syncthreads();
        if (warp != 0) return;
        float mm = lane < kScoreWarps ? s_m[lane] : -FLT_MAX;
        for (int o2 = 16; o2 > 0; o2 >>= 1) mm = fmaxf(mm, __shfl_xor_sync(0xffffffffu, mm, o2));
        double ss = lane < kScoreWarps ? (double)s_s[lane] * (double)expf(s_m[lane] - mm) : 0.0;
        for (int o2 = 16; o2 > 0; o2 >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o2);
        float lv[KC];
        uint32_t li[KC];
#pragma unroll
        for (int i = 0; i < KC; ++i) {
            lv[i] = lane < kScoreWarps ? s_v[lane][i] : -FLT_MAX;
            li[i] = lane < kScoreWarps ? s_i[lane][i] : 0xffffffffu;
        }
        warp_select<KC>(lv, li, lane, xv, ci);
        M = mm;
        S = (float)ss;
    }
    // ---- warp 0: rank by the exact order (all candidates are distinct rows) ----
    uint32_t rank = 0;
    for (int r = 0; r < KC; ++r) {
        const float ov = __shfl_sync(0xffffffffu, xv, r);
        const uint32_t oi = __shfl_sync(0xffffffffu, ci, r);
        if (lane < KC && (uint32_t)r != lane && better(ov, oi, xv, ci)) ++rank;
    }
    // exact maximum = the best candidate; both passes took the sum against it (M == best, the factor below is 1)
    float best = lane < KC ? xv : -FLT_MAX;
    for (int o2 = 16; o2 > 0; o2 >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o2));
    if (lane == 0) {
        o[0] = best;
        o[1] = S * __expf(M - best);
    }
    if (lane < KC) {
        if (ci == 0xffffffffu) rank = lane;   // fewer rows than candidates: the empty entries keep their places at the end
        o[2 + rank] = xv;
        o[2 + KC + rank] = __uint_as_float(ci);
    }
}

// One warp per sequence: merge the P partials, evaluate the k confidences, filter by residency, stage the requests;
// the last CTA compacts them in sequence order.
struct MergeArgs {
    const float* partials;
    uint32_t n_partials, batch, k;
    const uint32_t* req_ids;        // optional, per sequence
    uint32_t req_id, layer_id;
    const KvPageDev* pages;         // optional residency table
    uint64_t num_pages, va_base, timestamp;
    uint32_t* ids;                  // optional [batch][k]
    float* conf;                    // optional [batch][k]
    uint64_t* va;                   // optional [batch][k]
    speckv_prefetch_request_t* staged;   // [batch][k] scratch
    uint32_t* staged_count;              // [batch] scratch
    speckv_prefetch_request_t* table;    // optional: header + batch * k records
    speckv_prefetch_request_t* ring;     // optional: 16 most recent requests
    unsigned long long* total;           // requests emitted so far (prefetcher state shared by all calls)
    unsigned int* ticket;                // this call's "CTAs done" counter (zeroed by the hidden-state kernel)
    unsigned long long* call_count;      // optional (mapped host memory): this call's request count
};

template <int K>
__global__ void __launch_bounds__(kScoreThreads)
score_merge_kernel(const MergeArgs a) {
    constexpr int PW = 2 + 2 * K;
    __shared__ uint32_t s_scan[kScoreThreads];
    __shared__ bool s_last;
    const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t seq = blockIdx.x * kScoreWarps + warp;
    if (seq < a.batch) {
        float lv[K], mm = -FLT_MAX;
        uint32_t li[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            lv[k] = -FLT_MAX;
            li[k] = 0xffffffffu;
        }
        const float* base = a.partials + (size_t)seq * a.n_partials * PW;
        for (uint32_t p = lane; p < a.n_partials; p += 32) mm = fmaxf(mm, base[(size_t)p * PW]);
        for (int o = 16; o > 0; o >>= 1) mm = fmaxf(mm, __shfl_xor_sync(0xffffffffu, mm, o));
        // (fp32 exponentials and per-lane sums, the lanes combined in fp64: an fp32 tree over a few hundred partials of
        // similar size drifts by several ulps, which a confidence near 1/2 cannot afford; fp64 exp would cost this kernel
        // most of its time)
        float sl = 0.0f;   // a lane adds at most ceil(n_partials / 32) partials
        for (uint32_t p = lane; p < a.n_partials; p += 32) {
            const float* q = base + (size_t)p * PW;
            sl += q[1] * expf(q[0] - mm);
#pragma unroll
            for (int k = 0; k < K; ++k) list_insert<K>(lv, li, q[2 + k], __float_as_uint(q[2 + K + k]));
        }
        double ss = sl;
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        const float denom = (float)ss;
        // global top-k: k rounds of warp arg-max over the list heads, the winner pops its head
        float win_v = 0.0f;
        uint32_t win_i = 0;
        for (uint32_t r = 0; r < a.k; ++r) {
            float best = lv[0];
            uint32_t idx = li[0];
            for (int o = 16; o > 0; o >>= 1) {
                const float ob = __shfl_xor_sync(0xffffffffu, best, o);
                const uint32_t oi = __shfl_xor_sync(0xffffffffu, idx, o);
                if (better(ob, oi, best, idx)) {
                    best = ob;
                    idx = oi;
                }
            }
            if (li[0] == idx && idx != 0xffffffffu) {
#pragma unroll
                for (int i = 0; i + 1 < K; ++i) {
                    lv[i] = lv[i + 1];
                    li[i] = li[i + 1];
                }
                lv[K - 1] = -FLT_MAX;
                li[K - 1] = 0xffffffffu;
            }
            if (lane == r) {
                win_v = best;
                win_i = idx;
            }
        }
        // lanes 0 .. k-1 hold prediction i = lane
        bool keep = false;
        speckv_prefetch_request_t rq;
        if (lane < a.k) {
            const float e = expf(__fsub_rn(win_v, mm));
            const float cf = __fdiv_rn(e, denom);                                   // logits[i] /= sum_exp, :183-185
            const uint32_t rid = a.req_ids ? a.req_ids[seq] : a.req_id;
            const uint64_t va = ((uint64_t)rid << 32) | ((uint64_t)a.layer_id << 16) | (uint64_t)(lane + 1);
            const size_t o = (size_t)seq * a.k + lane;
            if (a.ids) a.ids[o] = win_i;
            if (a.conf) a.conf[o] = cf;
            if (a.va) a.va[o] = va;
            // already in L1 or L2 -> no request (speculative_prefetcher.cpp:51-54; is_in_cache, cxl_memory_manager.cpp:119-128)
            bool resident = false;
            if (a.pages && va >= a.va_base) {
                const uint64_t pi = (va - a.va_base) >> 12;
                if (pi < a.num_pages && __ldg(&a.pages[pi].virt_page_id) == (va & ~0xFFFULL))
                    resident = (__ldg(&a.pages[pi].flags) & 3u) != 0u;
            }
            keep = !resident;
            rq.virtual_addr = va;
            rq.layer_id = a.layer_id;
            rq.predicted_token_id = win_i;
            rq.confidence = cf;
            rq.reserved = 0;
            rq.timestamp = a.timestamp;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (keep) a.staged[(size_t)seq * a.k + __popc(bal & ((1u << lane) - 1u))] = rq;
        if (lane == 0) a.staged_count[seq] = (uint32_t)__popc(bal);
    }
    // ---- the last CTA compacts the staged requests in sequence order ----
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    uint32_t base = 0;
    for (uint32_t s0 = 0; s0 < a.batch; s0 += kScoreThreads) {
        const uint32_t s = s0 + tid;
        const uint32_t c = s < a.batch ? __ldcg(&a.staged_count[s]) : 0u;
        s_scan[tid] = c;
        __syncthreads();
        for (int o = 1; o < kScoreThreads; o <<= 1) {   // inclusive scan (Hillis-Steele; 256 entries, runs once per call)
            const uint32_t v = tid >= (uint32_t)o ? s_scan[tid - o] : 0u;
            __syncthreads();
            s_scan[tid] += v;
            __syncthreads();
        }
        const uint32_t off = base + s_scan[tid] - c;
        if (a.table)
            for (uint32_t i = 0; i < c; ++i) {
                const uint4* src = reinterpret_cast<const uint4*>(&a.staged[(size_t)s * a.k + i]);
                uint4* dst = reinterpret_cast<uint4*>(&a.table[1 + off + i]);
                dst[0] = __ldcg(src);
                dst[1] = __ldcg(src + 1);
            }
        base += s_scan[kScoreThreads - 1];
        __syncthreads();
    }
    const uint32_t n = base;
    __shared__ unsigned long long s_before;
    if (tid == 0) s_before = atomicAdd(a.total, (unsigned long long)n);
    __syncthreads();
    const unsigned long long before = s_before;
    if (a.table && tid == 0) {
        speckv_prefetch_request_t h;
        h.virtual_addr = n;                       // header: number of valid requests that follow
        h.layer_id = a.layer_id;
        h.predicted_token_id = a.batch * a.k;     // capacity
        h.confidence = 0.0f;
        h.reserved = 0;
        h.timestamp = a.timestamp;
        a.table[0] = h;
    }
    // outstanding queue: the 16 most recent requests stay visible (speculative_prefetcher.cpp:162-172)
    if (a.ring && a.table) {
        __syncthreads();
        const uint32_t keepn = min(n, kRing);
        if (tid < keepn) {
            const uint32_t i = n - keepn + tid;
            a.ring[(before + i) % kRing] = a.table[1 + i];
        }
    }
    if (tid == 0 && a.call_count) {
        *a.call_count = n;
        __threadfence_system();
    }
}

void free_predictor() {
    if (g_pred.d_emb) cudaFree(g_pred.d_emb);
    if (g_pred.d_wout) cudaFree(g_pred.d_wout);
    if (g_pred.d_rowsum) cudaFree(g_pred.d_rowsum);
    if (g_pred.d_cand) cudaFree(g_pred.d_cand);
    if (g_pred.d_ring) cudaFree(g_pred.d_ring);
    if (g_pred.d_total) cudaFree(g_pred.d_total);
    g_pred = Predictor();
}

// statistics of finished emit calls: total_prefetches += n and the reference's latency update
// (speculative_prefetcher.cpp:72-79: avg = (avg * (total - n) + latency_us) / total, total counted in requests)
void harvest_calls_locked(bool wait) {
    for (int i = 0; i < kEmitCalls; ++i) {
        EmitCall& c = g_calls[i];
        if (!c.busy) continue;
        const cudaError_t q = wait ? cudaEventSynchronize(c.b) : cudaEventQuery(c.b);
        if (q == cudaErrorNotReady) continue;
        float ms = 0.0f;
        if (q == cudaSuccess && cudaEventElapsedTime(&ms, c.a, c.b) == cudaSuccess) {
            const uint64_t n = g_h_counts ? (uint64_t)g_h_counts[i] : 0;
            g_stat_total += n;
            if (g_stat_total > 0)
                g_stat_latency_us = (g_stat_latency_us * (double)(g_stat_total - n) + (double)ms * 1e3) / (double)g_stat_total;
        } else {
            cudaGetLastError();
        }
        c.busy = false;
    }
}

// plan_only: n_partials and the dynamic shared memory the launch needs (smem), nothing launched
template <int K, int S>
cudaError_t launch_partial(uint32_t batch, const float* d_h, float* d_partials, uint32_t& n_partials, size_t& smem,
                           uint32_t plan_only, cudaStream_t st) {
    uint32_t seq_lanes = 4;   // at least 4: a tile (kScoreWarps * 32 / seq_lanes rows, double-buffered) must fit shared memory
    while (seq_lanes < 32 && seq_lanes * S < batch) seq_lanes <<= 1;
    const uint32_t nsub = kScoreWarps * (32u / seq_lanes);
    uint32_t rps = nsub >= 32 ? 1 : 32 / nsub;                       // tiles of >= 32 rows
    const uint32_t tile_rows = nsub * rps;
    const uint32_t n_tiles = (g_pred.vocab + tile_rows - 1) / tile_rows;
    const uint32_t sb = seq_lanes * S;
    const uint32_t gy = (batch + sb - 1) / sb;
    uint32_t gx = (uint32_t)current_sm_count() * 2u / (gy ? gy : 1u);
    if (gx < 1) gx = 1;
    if (gx > n_tiles) gx = n_tiles;
    n_partials = gx;
    constexpr int PW = 2 + 2 * K;
    const size_t tile_bytes = 2ull * tile_rows * tile_ld(g_pred.hidden) * sizeof(float);
    const size_t park_bytes = (size_t)nsub * sb * PW * sizeof(float);
    smem = tile_bytes > park_bytes ? tile_bytes : park_bytes;
    if (plan_only) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(score_partial_kernel<K, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    score_partial_kernel<K, S><<<dim3(gx, gy), kScoreThreads, smem, st>>>(g_pred.d_wout, g_pred.vocab, g_pred.hidden, d_h, batch,
                                                                         seq_lanes, rps, n_tiles, d_partials);
    return cudaGetLastError();
}

// the whole pipeline; any of ids / conf / va / table may be NULL
speckv_status_t score_emit(const uint32_t* d_tokens, uint32_t batch, uint32_t k, const uint32_t* d_req_ids, uint32_t req_id,
                           uint32_t layer_id, const speckv_page_t* d_pages, size_t num_pages, uint64_t va_base,
                           uint64_t timestamp, speckv_prefetch_request_t* d_table, uint32_t* d_ids, float* d_conf,
                           uint64_t* d_va, void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    std::lock_guard<std::mutex> lk(g_pred_mu);
    if (!g_pred.d_emb) return SPECKV_ERR_INVAL;   // no predictor loaded
    if (batch == 0) return SPECKV_OK;
    if (!d_tokens || k == 0 || k > (uint32_t)kMaxK || k > g_pred.vocab || (!d_pages && num_pages)) return SPECKV_ERR_INVAL;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != g_pred.device) return SPECKV_ERR_INVAL;   // weights live on another device
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    // rank-one scoring (candidates from h * rowsum[v], exact re-scoring) keeps k + 2 or more candidates; the tiled
    // exact kernel remains for k > 14 and for SPECKV_SCORE_EXACT=2 (=1: the rank-one kernel with exact logits only).
    // When a tile of W_out rows would not fit shared memory (wide hidden, small batches sooner), the rank-one kernel's
    // exact pass takes the tiled kernel's place: it reads W_out from global memory at any width, for any k <= 16.
    const char* ex_env = getenv("SPECKV_SCORE_EXACT");
    const int ex_mode = ex_env ? atoi(ex_env) : 0;
    bool rank1 = k <= 14 && ex_mode != 2;
    bool force_exact = ex_mode == 1;
    int KK = rank1 ? (k <= 6 ? 8 : 16) : (k <= 4 ? 4 : (k <= 8 ? 8 : 16));
    uint32_t n_partials = 1;
    size_t tile_smem = 0;
    cudaError_t e = cudaSuccess;
    if (!rank1) {
        e = KK == 4 ? launch_partial<4, 8>(batch, nullptr, nullptr, n_partials, tile_smem, 1, st)
          : KK == 8 ? launch_partial<8, 4>(batch, nullptr, nullptr, n_partials, tile_smem, 1, st)
                    : launch_partial<16, 2>(batch, nullptr, nullptr, n_partials, tile_smem, 1, st);
        if (tile_smem > g_pred.smem_optin) {
            rank1 = force_exact = true;
            KK = 16;
            n_partials = 1;
        }
    }
    const int PW = 2 + 2 * KK;
    // per-call scratch from the stream's persistent buffer (two calls on different streams never share it)
    const size_t off_h = 0, off_p = (((size_t)batch * 4) + 255) & ~(size_t)255;
    const size_t off_s = (off_p + (size_t)batch * n_partials * PW * 4 + 255) & ~(size_t)255;
    const size_t off_c = (off_s + (size_t)batch * k * sizeof(speckv_prefetch_request_t) + 255) & ~(size_t)255;
    const size_t off_t = (off_c + (size_t)batch * 4 + 255) & ~(size_t)255;
    const size_t total = off_t + 16;
    uint8_t* scratch = nullptr;
    if ((e = scratch_persistent((void**)&scratch, total, st)) != cudaSuccess) return status_of(e);
    float* d_h = reinterpret_cast<float*>(scratch + off_h);
    float* d_partials = reinterpret_cast<float*>(scratch + off_p);

    // statistics bracket (not while the stream is being captured into a graph)
    EmitCall* call = nullptr;
    int call_idx = -1;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (d_table && cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone) {
        for (int pass = 0; pass < 2 && !call; ++pass) {
            for (int i = 0; i < kEmitCalls; ++i)
                if (!g_calls[i].busy) {
                    call = &g_calls[i];
                    call_idx = i;
                    break;
                }
            if (!call) harvest_calls_locked(false);
        }
        if (call && !call->a && (cudaEventCreate(&call->a) != cudaSuccess || cudaEventCreate(&call->b) != cudaSuccess)) {
            cudaGetLastError();
            call = nullptr;
        }
        if (call) {
            call->busy = true;
            cudaEventRecord(call->a, st);
        }
    } else {
        cudaGetLastError();
    }

    const uint32_t nj = g_pred.emb_dim < g_pred.hidden ? g_pred.emb_dim : g_pred.hidden;
    const size_t hsmem = (size_t)kHiddenWarps * g_pred.hist_len * nj * sizeof(float);
    if (hsmem <= 48 * 1024)
        hidden_warp_kernel<<<(batch + kHiddenWarps - 1) / kHiddenWarps, kHiddenWarps * 32, hsmem, st>>>(
            d_tokens, batch, g_pred.hist_len, g_pred.d_emb, g_pred.vocab, g_pred.emb_dim, g_pred.hidden, g_pred.layers, d_h,
            reinterpret_cast<unsigned int*>(scratch + off_t));
    else
        hidden_kernel<<<(batch + 127) / 128, 128, 0, st>>>(d_tokens, batch, g_pred.hist_len, g_pred.d_emb, g_pred.vocab,
                                                           g_pred.emb_dim, g_pred.hidden, g_pred.layers, d_h,
                                                           reinterpret_cast<unsigned int*>(scratch + off_t));
    if (rank1) {
        if (KK == 8)
            score_rank1_kernel<8><<<batch, kScoreThreads, 0, st>>>(g_pred.d_wout, g_pred.d_rowsum, g_pred.d_cand, g_pred.vocab, g_pred.hidden, d_h,
                                                                  batch, k, g_pred.row_abs_max, force_exact, d_partials);
        else
            score_rank1_kernel<16><<<batch, kScoreThreads, 0, st>>>(g_pred.d_wout, g_pred.d_rowsum, g_pred.d_cand, g_pred.vocab, g_pred.hidden, d_h,
                                                                   batch, k, g_pred.row_abs_max, force_exact, d_partials);
        e = cudaGetLastError();
    } else {
        e = KK == 4 ? launch_partial<4, 8>(batch, d_h, d_partials, n_partials, tile_smem, 0, st)
          : KK == 8 ? launch_partial<8, 4>(batch, d_h, d_partials, n_partials, tile_smem, 0, st)
                    : launch_partial<16, 2>(batch, d_h, d_partials, n_partials, tile_smem, 0, st);
    }
    if (e != cudaSuccess) return status_of(e);
    MergeArgs m;
    m.partials = d_partials;
    m.n_partials = n_partials;
    m.batch = batch;
    m.k = k;
    m.req_ids = d_req_ids;
    m.req_id = req_id;
    m.layer_id = layer_id;
    m.pages = reinterpret_cast<const KvPageDev*>(d_pages);
    m.num_pages = num_pages;
    m.va_base = va_base;
    m.timestamp = timestamp;
    m.ids = d_ids;
    m.conf = d_conf;
    m.va = d_va;
    m.staged = reinterpret_cast<speckv_prefetch_request_t*>(scratch + off_s);
    m.staged_count = reinterpret_cast<uint32_t*>(scratch + off_c);
    m.table = d_table;
    m.ring = g_pred.d_ring;
    m.total = g_pred.d_total;
    m.ticket = reinterpret_cast<unsigned int*>(scratch + off_t);
    m.call_count = (call && g_d_counts) ? g_d_counts + call_idx : nullptr;
    const unsigned grid = (batch + kScoreWarps - 1) / kScoreWarps;
    if (KK == 4) score_merge_kernel<4><<<grid, kScoreThreads, 0, st>>>(m);
    else if (KK == 8) score_merge_kernel<8><<<grid, kScoreThreads, 0, st>>>(m);
    else score_merge_kernel<16><<<grid, kScoreThreads, 0, st>>>(m);
    count_launch(3);
    if (call) cudaEventRecord(call->b, st);
    return status_of(cudaGetLastError());
}

}  // namespace
}  // namespace speckv

using namespace speckv;

extern "C" {

speckv_status_t speckv_ext_predictor_load(const float* h_embedding, const float* h_output, uint32_t vocab,
                                          uint32_t emb_dim, uint32_t hidden, uint32_t layers, uint32_t history_len) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if (!h_embedding || !h_output || !vocab || !emb_dim || !hidden || !history_len) return SPECKV_ERR_INVAL;
    // the rank-one kernel stages candidate rows in chunks and the tiled kernel's tile is checked per call (too wide a
    // tile falls back to the rank-one exact pass), so no width is unscorable; 4096 bounds the per-row work of a thread
    if (hidden > 4096) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(g_pred_mu);
    harvest_calls_locked(true);
    free_predictor();
    cudaError_t e = cudaGetDevice(&g_pred.device);
    int optin = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, g_pred.device);
    g_pred.smem_optin = (size_t)optin;
    if (e == cudaSuccess) e = cudaMalloc((void**)&g_pred.d_emb, (size_t)vocab * emb_dim * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc((void**)&g_pred.d_wout, (size_t)vocab * hidden * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc((void**)&g_pred.d_ring, kRing * sizeof(speckv_prefetch_request_t));
    if (e == cudaSuccess) e = cudaMalloc((void**)&g_pred.d_total, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(g_pred.d_ring, 0, kRing * sizeof(speckv_prefetch_request_t));
    if (e == cudaSuccess) e = cudaMemset(g_pred.d_total, 0, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemcpy(g_pred.d_emb, h_embedding, (size_t)vocab * emb_dim * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(g_pred.d_wout, h_output, (size_t)vocab * hidden * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        // rank-one form of the logits: row sums (fp64, rounded once) and the largest absolute row sum for its error bound
        std::vector<float> rs(vocab);
        double amax = 0.0;
        for (uint32_t v = 0; v < vocab; ++v) {
            const float* w = h_output + (size_t)v * hidden;
            double sum = 0.0, asum = 0.0;
            for (uint32_t j = 0; j < hidden; ++j) {
                sum += (double)w[j];
                asum += fabs((double)w[j]);
            }
            rs[v] = (float)sum;
            if (!(asum <= amax)) amax = asum;   // a NaN row makes the bound NaN: every sequence then takes the exact pass
        }
        g_pred.row_abs_max = nextafterf((float)amax, INFINITY);
        e = cudaMalloc((void**)&g_pred.d_rowsum, (size_t)vocab * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpy(g_pred.d_rowsum, rs.data(), (size_t)vocab * sizeof(float), cudaMemcpyHostToDevice);
        // candidate orders (ties by the lower id in both, as the final ranking does); NaN sums sort last and make the bound NaN
        std::vector<uint32_t> idx(vocab), cand(2 * 16, 0u);
        for (uint32_t v = 0; v < vocab; ++v) idx[v] = v;
        const size_t nc = vocab < 16u ? vocab : 16u;
        for (int dir = 0; dir < 2; ++dir) {
            auto key = [&](uint32_t v) { return rs[v] != rs[v] ? -INFINITY : (dir ? -rs[v] : rs[v]); };
            std::partial_sort(idx.begin(), idx.begin() + nc, idx.end(), [&](uint32_t a, uint32_t b) {
                const float ka = key(a), kb = key(b);
                return ka > kb || (ka == kb && a < b);
            });
            for (size_t i = 0; i < nc; ++i) cand[16 * dir + i] = idx[i];
        }
        if (e == cudaSuccess) e = cudaMalloc((void**)&g_pred.d_cand, cand.size() * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMemcpy(g_pred.d_cand, cand.data(), cand.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess && !g_h_counts) {
        e = cudaHostAlloc((void**)&g_h_counts, kEmitCalls * sizeof(unsigned long long), cudaHostAllocMapped | cudaHostAllocPortable);
        if (e == cudaSuccess) e = cudaHostGetDevicePointer((void**)&g_d_counts, g_h_counts, 0);
        if (e != cudaSuccess) {   // statistics only: go on without the per-call counts
            cudaGetLastError();
            g_h_counts = g_d_counts = nullptr;
            e = cudaSuccess;
        }
    }
    if (e != cudaSuccess) {
        free_predictor();
        return status_of(e);
    }
    g_pred.vocab = vocab;
    g_pred.emb_dim = emb_dim;
    g_pred.hidden = hidden;
    g_pred.layers = layers;
    g_pred.hist_len = history_len;
    g_stat_total = g_stat_mispred = 0;
    g_stat_latency_us = 0.0;
    return SPECKV_OK;
}

void speckv_ext_predictor_unload(void) {
    std::lock_guard<std::mutex> lk(g_pred_mu);
    if (device_count() > 0) {
        harvest_calls_locked(true);
        free_predictor();
    }
}

speckv_status_t speckv_ext_prefetch_score(const uint32_t* d_tokens, uint32_t batch, uint32_t k, uint32_t req_id,
                                          uint32_t layer_id, uint32_t* d_ids, float* d_conf, uint64_t* d_va,
                                          void* cuda_stream) {
    if (batch && (!d_ids || !d_conf || !d_va)) return device_count() <= 0 ? SPECKV_ERR_DRIVER : SPECKV_ERR_INVAL;
    return score_emit(d_tokens, batch, k, nullptr, req_id, layer_id, nullptr, 0, 0, 0, nullptr, d_ids, d_conf, d_va, cuda_stream);
}

speckv_status_t speckv_ext_prefetch_emit(const uint32_t* d_tokens, uint32_t batch, uint32_t k, const uint32_t* d_req_ids,
                                         uint32_t req_id, uint32_t layer_id, const speckv_page_t* d_pages, size_t num_pages,
                                         uint64_t va_base, uint64_t timestamp, speckv_prefetch_request_t* d_table,
                                         uint32_t* d_ids, float* d_conf, void* cuda_stream) {
    if (batch && !d_table) return device_count() <= 0 ? SPECKV_ERR_DRIVER : SPECKV_ERR_INVAL;
    return score_emit(d_tokens, batch, k, d_req_ids, req_id, layer_id, d_pages, num_pages, va_base, timestamp, d_table, d_ids,
                      d_conf, nullptr, cuda_stream);
}

// SpeculativePrefetcher::handle_misprediction (speculative_prefetcher.cpp:84-97): the counter moves only when the
// actual token is not among the predicted ones.  Host logic.
speckv_status_t speckv_ext_prefetch_handle_misprediction(uint32_t actual_token, const uint32_t* h_predicted, size_t n,
                                                         int* out_was_correct) {
    if (!h_predicted && n) return SPECKV_ERR_INVAL;
    bool ok = false;
    for (size_t i = 0; i < n; ++i) ok |= h_predicted[i] == actual_token;
    std::lock_guard<std::mutex> lk(g_pred_mu);
    if (!ok) ++g_stat_mispred;
    if (out_was_correct) *out_was_correct = ok ? 1 : 0;
    return SPECKV_OK;
}

// SpeculativePrefetcher::get_statistics (speculative_prefetcher.cpp:126-137).  successful_prefetches is never
// incremented anywhere in the reference, so hit_rate and precision are 0 there as well.
speckv_status_t speckv_ext_prefetch_stats(speckv_prefetch_stats_t* out, int reset) {
    if (!out) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(g_pred_mu);
    if (device_count() > 0) harvest_calls_locked(true);
    out->total_prefetches = g_stat_total;
    out->successful_prefetches = 0;
    out->mispredictions = g_stat_mispred;
    out->hit_rate = 0.0;
    out->precision = 0.0;
    if (out->total_prefetches > 0) {
        out->hit_rate = (double)out->successful_prefetches / (double)out->total_prefetches;
        out->precision = (double)out->successful_prefetches / (double)(out->successful_prefetches + out->mispredictions + 1);
    }
    out->avg_prediction_latency_us = g_stat_latency_us;
    if (reset) {   // reset_statistics, :139-142
        g_stat_total = g_stat_mispred = 0;
        g_stat_latency_us = 0.0;
    }
    return SPECKV_OK;
}

// SpeculativePrefetcher::is_already_prefetched (speculative_prefetcher.cpp:174-185) over the device-side queue of the
// 16 most recent requests; copies the queue to the host (oldest first) when h_queue is given.  Blocking.
speckv_status_t speckv_ext_prefetch_outstanding(const uint64_t* h_va, size_t n, uint8_t* out_found,
                                                speckv_prefetch_request_t* h_queue, uint32_t* out_queue_len,
                                                void* cuda_stream) {
    if (device_count() <= 0) return SPECKV_ERR_DRIVER;
    if ((!h_va || !out_found) && n) return SPECKV_ERR_INVAL;
    std::lock_guard<std::mutex> lk(g_pred_mu);
    if (!g_pred.d_ring) return SPECKV_ERR_INVAL;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    speckv_prefetch_request_t ring[kRing];
    unsigned long long tot[1] = {0};
    cudaError_t e = cudaMemcpyAsync(ring, g_pred.d_ring, sizeof(ring), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(tot, g_pred.d_total, sizeof(tot), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return status_of(e);
    const uint32_t len = tot[0] < kRing ? (uint32_t)tot[0] : kRing;
    for (size_t i = 0; i < n; ++i) {
        out_found[i] = 0;
        for (uint32_t q = 0; q < len; ++q)
            if (ring[(tot[0] - len + q) % kRing].virtual_addr == h_va[i]) out_found[i] = 1;
    }
    if (h_queue)
        for (uint32_t q = 0; q < len; ++q) h_queue[q] = ring[(tot[0] - len + q) % kRing];
    if (out_queue_len) *out_queue_len = len;
    return SPECKV_OK;
}

}  // extern "C"
