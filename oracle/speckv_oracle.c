/*
 * speckv_oracle.c -- CPU restatement of the CXL-SpecKV cache-engine hot path.
 *
 * TEST INFRASTRUCTURE ONLY (see speckv_oracle.h).  Parity status: PINNED
 * against oracle/_ref (the reference's own sources compiled unmodified) and
 * the fixtures in tests/golden/.
 *
 * Build: gcc -O2 -fPIC -shared -ffp-contract=off (never -ffast-math: it changes
 * the bitstream, SURVEY.md section 8c) -pthread -lm.
 *
 * Every function cites the reference lines it follows (/root/reference/...).
 */
#include "speckv_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------ */
/* fp16 / bf16 boundary                                                      */
/* ------------------------------------------------------------------------ */

float oracle_widen(uint16_t bits, int dtype) {
    if (dtype == ORACLE_BF16) {
        uint32_t u = (uint32_t)bits << 16;
        float f;
        memcpy(&f, &u, 4);
        return f;
    }
    _Float16 h;
    memcpy(&h, &bits, 2);
    return (float)h; /* exact */
}

uint16_t oracle_narrow(float v, int dtype) {
    uint16_t out;
    if (dtype == ORACLE_BF16) {
        uint32_t u;
        memcpy(&u, &v, 4);
        if ((u & 0x7fffffffu) > 0x7f800000u) { /* NaN: keep quiet NaN, sign */
            return (uint16_t)((u >> 16) | 0x0040u);
        }
        uint32_t lsb = (u >> 16) & 1u;
        u += 0x7fffu + lsb; /* round to nearest even */
        return (uint16_t)(u >> 16);
    }
    _Float16 h = (_Float16)v; /* RN-even */
    memcpy(&out, &h, 2);
    return out;
}

/* ------------------------------------------------------------------------ */
/* compression: src/fpga_engine/cache_engine.cpp                             */
/* ------------------------------------------------------------------------ */

/* compute_scale_factor, cache_engine.cpp:172-184.  `abs_val > max_val` skips
 * NaN; all-zero (or all-NaN) input gives scale 1.0f. */
float oracle_scale(const float* x, size_t n) {
    float max_val = 0.0f;
    for (size_t i = 0; i < n; ++i) {
        float a = fabsf(x[i]);
        if (a > max_val) max_val = a;
    }
    return (max_val > 0.0f) ? (max_val / 127.0f) : 1.0f;
}

/* static_cast<int8_t>(float) as x86-64 GCC performs it (cvttss2si to a 32-bit
 * register, then the low byte): out-of-range and NaN become 0x80000000, whose
 * low byte is 0.  cache_engine.cpp:191; the clamp at :192 is dead code because
 * its operand is already an int8_t. */
static inline int8_t cast_float_to_i8(float r) {
    int32_t t;
    if (!(fabsf(r) < 2147483648.0f)) t = INT32_MIN; /* also catches NaN */
    else t = (int32_t)r;
    return (int8_t)(uint8_t)((uint32_t)t & 0xffu);
}

/* quantize_to_int8, cache_engine.cpp:186-196: q = int8(round((x/s)*127)),
 * round = std::round = half away from zero.  x/s is already in [-127,127]
 * so the second *127 makes the code wrap modulo 256 (SURVEY.md fact 1). */
void oracle_quantize(const float* x, size_t n, float scale, int8_t* q) {
    for (size_t i = 0; i < n; ++i) {
        float scaled = x[i] / scale;
        q[i] = cast_float_to_i8(roundf(scaled * 127.0f));
    }
}

/* delta_encode, cache_engine.cpp:198-211 (int8 arithmetic wraps mod 256) */
void oracle_delta_encode(const int8_t* q, size_t n, int8_t* d) {
    if (n == 0) return;
    d[0] = q[0];
    for (size_t i = 1; i < n; ++i) d[i] = (int8_t)(uint8_t)((uint8_t)q[i] - (uint8_t)q[i - 1]);
}

/* run_length_encode, cache_engine.cpp:213-239: [value][count] byte pairs,
 * a run is cut when count reaches 255. */
size_t oracle_rle_encode(const int8_t* d, size_t n, uint8_t* out) {
    if (n == 0) return 0;
    size_t w = 0;
    int8_t cur = d[0];
    size_t count = 1;
    for (size_t i = 1; i < n; ++i) {
        if (d[i] == cur && count < 255) {
            count++;
        } else {
            out[w++] = (uint8_t)cur;
            out[w++] = (uint8_t)count;
            cur = d[i];
            count = 1;
        }
    }
    out[w++] = (uint8_t)cur;
    out[w++] = (uint8_t)count;
    return w;
}

/* FPGACacheEngine::compress, cache_engine.cpp:40-82.  num_tokens, hidden_dim
 * and layer_id are ignored by the reference (only kv_data.size() matters). */
size_t oracle_compress(const float* x, size_t n, float* scale, uint8_t* out) {
    float s = oracle_scale(x, n);
    *scale = s;
    if (n == 0) return 0;
    int8_t* q = (int8_t*)malloc(n);
    int8_t* d = (int8_t*)malloc(n);
    oracle_quantize(x, n, s, q);
    oracle_delta_encode(q, n, d);
    size_t bytes = oracle_rle_encode(d, n, out);
    free(q);
    free(d);
    return bytes;
}

/* run_length_decode, cache_engine.cpp:241-258: a trailing odd byte is ignored,
 * a pair with count 0 emits nothing.  Stops at cap (the reference grows a vector). */
size_t oracle_rle_decode(const uint8_t* rle, size_t bytes, int8_t* out, size_t cap) {
    size_t n = 0;
    for (size_t i = 0; i + 1 < bytes; i += 2) {
        int8_t v = (int8_t)rle[i];
        uint8_t c = rle[i + 1];
        for (size_t j = 0; j < c; ++j) {
            if (n >= cap) return n;
            out[n++] = v;
        }
    }
    return n;
}

/* delta_decode, cache_engine.cpp:260-273 */
void oracle_delta_decode(const int8_t* d, size_t n, int8_t* q) {
    if (n == 0) return;
    q[0] = d[0];
    for (size_t i = 1; i < n; ++i) q[i] = (int8_t)(uint8_t)((uint8_t)q[i - 1] + (uint8_t)d[i]);
}

/* dequantize_from_int8, cache_engine.cpp:275-284 */
void oracle_dequantize(const int8_t* q, size_t n, float scale, float* y) {
    for (size_t i = 0; i < n; ++i) {
        float scaled = (float)q[i] / 127.0f;
        y[i] = scaled * scale;
    }
}

/* FPGACacheEngine::decompress, cache_engine.cpp:84-116 */
size_t oracle_decompress(const uint8_t* rle, size_t bytes, float scale, float* out, size_t cap) {
    if (cap == 0) return 0;
    int8_t* d = (int8_t*)malloc(cap);
    int8_t* q = (int8_t*)malloc(cap);
    size_t n = oracle_rle_decode(rle, bytes, d, cap);
    oracle_delta_decode(d, n, q);
    oracle_dequantize(q, n, scale, out);
    free(d);
    free(q);
    return n;
}

/* ------------------------------------------------------------------------ */
/* the other compression schemes                                             */
/* ------------------------------------------------------------------------ */
/* Scheme 1 (SPECKV_COMP_INT8, host/include/speckv.h:61) is the reference's quantiser on its own: the codes of
 * quantize_to_int8 (:186-196), one byte per element, decoded by dequantize_from_int8 (:275-284).
 *
 * Schemes 3 and 4 are NOT reference behaviour (SURVEY.md section 8f-4 asks for them as explicit new ids): the
 * reference multiplies by 127 twice -- s = max / 127 (:183) and (x / s) * 127 (:190-191) -- so its codes wrap modulo
 * 256 and the clamp at :192 is dead.  The clamped schemes keep every operation of :186-196 and :275-284, apply the
 * clamp BEFORE the narrowing cast as :192 intended, and store s = max|x| so that (x / s) * 127 spans [-127, 127]:
 * quantiser and dequantiser become inverse to each other.  NaN codes as 0.  Scheme 3 = clamped codes + delta + RLE,
 * scheme 4 = clamped codes only. */
float oracle_scale_max(const float* x, size_t n) {
    float max_val = 0.0f;
    for (size_t i = 0; i < n; ++i) {
        float a = fabsf(x[i]);
        if (a > max_val) max_val = a;
    }
    return (max_val > 0.0f) ? max_val : 1.0f;
}

void oracle_quantize_clamped(const float* x, size_t n, float scale, int8_t* q) {
    for (size_t i = 0; i < n; ++i) {
        float r = roundf((x[i] / scale) * 127.0f);
        int v = (r != r) ? 0 : (r > 127.0f ? 127 : (r < -128.0f ? -128 : (int)r));
        q[i] = (int8_t)v;
    }
}

size_t oracle_compress_scheme(const float* x, size_t n, int scheme, float* scale, uint8_t* out) {
    if (scheme == ORACLE_SCHEME_RLE) return oracle_compress(x, n, scale, out);
    const int clamped = scheme == ORACLE_SCHEME_CLAMP_RLE || scheme == ORACLE_SCHEME_CLAMP_INT8;
    float s = clamped ? oracle_scale_max(x, n) : oracle_scale(x, n);
    *scale = s;
    if (n == 0) return 0;
    int8_t* q = (int8_t*)malloc(n);
    if (clamped) oracle_quantize_clamped(x, n, s, q);
    else oracle_quantize(x, n, s, q);
    size_t bytes;
    if (scheme == ORACLE_SCHEME_CLAMP_RLE) {
        int8_t* d = (int8_t*)malloc(n);
        oracle_delta_encode(q, n, d);
        bytes = oracle_rle_encode(d, n, out);
        free(d);
    } else {
        memcpy(out, q, n);
        bytes = n;
    }
    free(q);
    return bytes;
}

size_t oracle_decompress_scheme(const uint8_t* payload, size_t bytes, float scale, int scheme, float* out, size_t cap) {
    if (scheme == ORACLE_SCHEME_RLE || scheme == ORACLE_SCHEME_CLAMP_RLE) return oracle_decompress(payload, bytes, scale, out, cap);
    size_t n = bytes < cap ? bytes : cap;
    oracle_dequantize((const int8_t*)payload, n, scale, out);
    return n;
}

/* ------------------------------------------------------------------------ */
/* batched forms (independent groups; optional pthread fan-out)              */
/* ------------------------------------------------------------------------ */

typedef struct {
    int is_compress;
    int scheme;            /* ORACLE_SCHEME_* */
    const void* in;
    int dtype;
    size_t group_elems, g0, g1;
    uint8_t* payload;
    const uint8_t* cpayload;
    size_t slot_bytes;
    float* scales;
    const float* cscales;
    uint32_t* comp_bytes;
    const uint32_t* ccomp_bytes;
    void* out;
    uint32_t* out_elems;
} batch_job_t;

static size_t elem_size(int dtype) { return dtype == ORACLE_F32 ? 4 : 2; }

static void* batch_worker(void* arg) {
    batch_job_t* j = (batch_job_t*)arg;
    size_t n = j->group_elems;
    float* tmp = (float*)malloc((n ? n : 1) * sizeof(float));
    uint8_t* buf = (uint8_t*)malloc(2 * (n ? n : 1));
    for (size_t g = j->g0; g < j->g1; ++g) {
        if (j->is_compress) {
            const float* x;
            if (j->dtype == ORACLE_F32) {
                x = (const float*)j->in + g * n;
            } else {
                const uint16_t* src = (const uint16_t*)j->in + g * n;
                for (size_t i = 0; i < n; ++i) tmp[i] = oracle_widen(src[i], j->dtype);
                x = tmp;
            }
            float s;
            size_t bytes = oracle_compress_scheme(x, n, j->scheme, &s, buf);
            size_t w = bytes < j->slot_bytes ? bytes : j->slot_bytes;
            memcpy(j->payload + g * j->slot_bytes, buf, w);
            j->scales[g] = s;
            j->comp_bytes[g] = (uint32_t)bytes;
        } else {
            size_t got = oracle_decompress_scheme(j->cpayload + g * j->slot_bytes, j->ccomp_bytes[g],
                                                  j->cscales[g], j->scheme, tmp, n);
            if (j->dtype == ORACLE_F32) {
                memcpy((float*)j->out + g * n, tmp, got * sizeof(float));
            } else {
                uint16_t* dst = (uint16_t*)j->out + g * n;
                for (size_t i = 0; i < got; ++i) dst[i] = oracle_narrow(tmp[i], j->dtype);
            }
            if (j->out_elems) j->out_elems[g] = (uint32_t)got;
        }
    }
    free(tmp);
    free(buf);
    return NULL;
}

static int run_batch(batch_job_t* proto, size_t n_groups, int threads) {
    if (threads < 1) threads = 1;
    if ((size_t)threads > n_groups) threads = n_groups ? (int)n_groups : 1;
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * threads);
    batch_job_t* jobs = (batch_job_t*)malloc(sizeof(batch_job_t) * threads);
    size_t per = (n_groups + threads - 1) / threads;
    for (int t = 0; t < threads; ++t) {
        jobs[t] = *proto;
        jobs[t].g0 = (size_t)t * per < n_groups ? (size_t)t * per : n_groups;
        jobs[t].g1 = (size_t)(t + 1) * per < n_groups ? (size_t)(t + 1) * per : n_groups;
        if (threads == 1) batch_worker(&jobs[t]);
        else pthread_create(&th[t], NULL, batch_worker, &jobs[t]);
    }
    if (threads > 1)
        for (int t = 0; t < threads; ++t) pthread_join(th[t], NULL);
    free(th);
    free(jobs);
    return 0;
}

int oracle_compress_batch(const void* in, int dtype, size_t group_elems, size_t n_groups,
                          uint8_t* payload, size_t slot_bytes, float* scales,
                          uint32_t* comp_bytes, int threads) {
    return oracle_compress_batch_scheme(in, dtype, group_elems, n_groups, payload, slot_bytes, scales, comp_bytes,
                                        ORACLE_SCHEME_RLE, threads);
}

int oracle_compress_batch_scheme(const void* in, int dtype, size_t group_elems, size_t n_groups,
                                 uint8_t* payload, size_t slot_bytes, float* scales,
                                 uint32_t* comp_bytes, int scheme, int threads) {
    (void)elem_size;
    batch_job_t j;
    memset(&j, 0, sizeof(j));
    j.is_compress = 1;
    j.scheme = scheme;
    j.in = in;
    j.dtype = dtype;
    j.group_elems = group_elems;
    j.payload = payload;
    j.slot_bytes = slot_bytes;
    j.scales = scales;
    j.comp_bytes = comp_bytes;
    return run_batch(&j, n_groups, threads);
}

int oracle_decompress_batch(const uint8_t* payload, size_t slot_bytes, const float* scales,
                            const uint32_t* comp_bytes, size_t group_elems, size_t n_groups,
                            int dtype, void* out, uint32_t* out_elems, int threads) {
    return oracle_decompress_batch_scheme(payload, slot_bytes, scales, comp_bytes, group_elems, n_groups, dtype, out,
                                          out_elems, ORACLE_SCHEME_RLE, threads);
}

int oracle_decompress_batch_scheme(const uint8_t* payload, size_t slot_bytes, const float* scales,
                                   const uint32_t* comp_bytes, size_t group_elems, size_t n_groups,
                                   int dtype, void* out, uint32_t* out_elems, int scheme, int threads) {
    batch_job_t j;
    memset(&j, 0, sizeof(j));
    j.is_compress = 0;
    j.scheme = scheme;
    j.dtype = dtype;
    j.group_elems = group_elems;
    j.cpayload = payload;
    j.slot_bytes = slot_bytes;
    j.cscales = scales;
    j.ccomp_bytes = comp_bytes;
    j.out = out;
    j.out_elems = out_elems;
    return run_batch(&j, n_groups, threads);
}

/* ------------------------------------------------------------------------ */
/* address translation                                                       */
/* ------------------------------------------------------------------------ */

/* page_walk, address_translation.cpp:85-90; same formula on the engine's miss
 * path, cache_engine.cpp:132.  A TLB hit returns entry.pa + offset where
 * entry.pa = pa & ~0xFFF of the filling miss (:136, address_translation.cpp:42)
 * i.e. the same value. */
uint64_t oracle_translate(uint64_t va) {
    return 0x4000000000ULL + (va & 0xFFFFFFFFFFFFULL);
}

oracle_atu_t* oracle_atu_new(size_t tlb_size) {
    oracle_atu_t* a = (oracle_atu_t*)calloc(1, sizeof(*a));
    a->size = tlb_size;
    a->vpage = (uint64_t*)calloc(tlb_size, 8);
    a->ppage = (uint64_t*)calloc(tlb_size, 8);
    a->valid = (uint8_t*)calloc(tlb_size, 1);
    return a;
}

void oracle_atu_free(oracle_atu_t* a) {
    if (!a) return;
    free(a->vpage);
    free(a->ppage);
    free(a->valid);
    free(a);
}

/* AddressTranslationUnit::translate, address_translation.cpp:19-46 */
uint64_t oracle_atu_translate(oracle_atu_t* a, uint64_t va) {
    uint64_t vpage = va & ~0xFFFULL;
    uint64_t off = va & 0xFFFULL;
    size_t idx = (size_t)((vpage >> 12) % a->size);
    if (a->valid[idx] && a->vpage[idx] == vpage) {
        a->hits++;
        return a->ppage[idx] + off;
    }
    a->misses++;
    uint64_t pa = oracle_translate(va); /* page_walk(virtual_addr): takes the full va */
    a->vpage[idx] = vpage;
    a->ppage[idx] = pa & ~0xFFFULL;
    a->valid[idx] = 1;
    return pa + off; /* :45 adds the offset again on the miss path */
}

/* invalidate, address_translation.cpp:48-58 (note: does not test `valid`) */
void oracle_atu_invalidate(oracle_atu_t* a, uint64_t va) {
    uint64_t vpage = va & ~0xFFFULL;
    size_t idx = (size_t)((vpage >> 12) % a->size);
    if (a->vpage[idx] == vpage) a->valid[idx] = 0;
}

void oracle_atu_invalidate_all(oracle_atu_t* a) { memset(a->valid, 0, a->size); }

void oracle_atu_stats(const oracle_atu_t* a, uint64_t* hits, uint64_t* misses) {
    *hits = a->hits;
    *misses = a->misses;
}

/* ------------------------------------------------------------------------ */
/* host page-table formulas: host/src/speckv_allocator.cpp                   */
/* ------------------------------------------------------------------------ */

uint64_t oracle_virt_page_id(uint64_t handle, uint64_t i) { return (handle << 32) | (i << 12); }       /* :24 */
uint64_t oracle_phys_page_id(uint64_t handle, uint64_t i) {                                           /* :25 */
    return 0x4000000000ULL + (handle << 20) + (i << 12);
}

/* SpeckvAllocator::access :54-74 (0 == nullptr == error at the C API) */
uint64_t oracle_access_addr(uint64_t handle, uint64_t alloc_bytes, uint64_t offset) {
    uint64_t num_pages = (alloc_bytes + 4095) / 4096; /* :19 */
    uint64_t page_idx = offset / 4096, page_off = offset % 4096;
    if (page_idx >= num_pages) return 0;
    return oracle_phys_page_id(handle, page_idx) + page_off;
}

uint64_t oracle_fetch_gpu_addr(uint64_t virt_page_id) {                                               /* :124 */
    return 0x8000000000ULL + (virt_page_id & 0xFFFFFFFFFFFFULL);
}

/* ------------------------------------------------------------------------ */
/* LSTM prefetch scoring: src/prefetcher/lstm_predictor.cpp                  */
/* ------------------------------------------------------------------------ */

void oracle_lstm_init_weights(unsigned seed, float* emb, size_t n_emb, float* lstm, size_t n_lstm,
                              float* wout, size_t n_out) {
    srand(seed); /* the reference never seeds: glibc default == srand(1) */
    for (size_t i = 0; i < n_emb; ++i) emb[i] = ((float)rand() / RAND_MAX - 0.5f) * 0.1f;   /* :27-29 */
    for (size_t i = 0; i < n_lstm; ++i) {                                                   /* :30-32 */
        float w = ((float)rand() / RAND_MAX - 0.5f) * 0.1f;
        if (lstm) lstm[i] = w;
    }
    for (size_t i = 0; i < n_out; ++i) wout[i] = ((float)rand() / RAND_MAX - 0.5f) * 0.1f;  /* :33-35 */
}

void oracle_lstm_predict_topk(const float* emb, const float* wout,
                              size_t vocab, size_t emb_dim, size_t hidden, size_t layers,
                              size_t hist_len, const uint32_t* hist_in, size_t n_hist, size_t k,
                              uint32_t* ids, float* conf, float* hidden_out) {
    /* history window, :46-51: keep the last hist_len, left-pad with token 0 */
    uint32_t* hist = (uint32_t*)calloc(hist_len ? hist_len : 1, sizeof(uint32_t));
    if (n_hist >= hist_len) {
        memcpy(hist, hist_in + (n_hist - hist_len), hist_len * sizeof(uint32_t));
    } else {
        memcpy(hist + (hist_len - n_hist), hist_in, n_hist * sizeof(uint32_t));
    }
    float* h = (float*)calloc(hidden, sizeof(float));
    float* c = (float*)calloc(hidden, sizeof(float));
    float* e = (float*)calloc(emb_dim, sizeof(float));
    for (size_t t = 0; t < hist_len; ++t) {
        /* embed_token :149-160: out-of-vocabulary ids embed to zeros */
        for (size_t j = 0; j < emb_dim; ++j) e[j] = 0.0f;
        if (hist[t] < vocab)
            for (size_t j = 0; j < emb_dim; ++j) e[j] = emb[(size_t)hist[t] * emb_dim + j];
        /* lstm_forward :116-147, called once per layer with the SAME embedded
         * input and state; the per-layer weight slice is copied and ignored. */
        for (size_t layer = 0; layer < layers; ++layer) {
            for (size_t i = 0; i < hidden; ++i) {
                float g = 0.0f;
                for (size_t j = 0; j < emb_dim && j < hidden; ++j) g += e[j] * 0.1f; /* :138-140 */
                c[i] = 0.5f * c[i] + 0.5f * tanhf(g);                                /* :143 */
                h[i] = 0.5f * tanhf(c[i]);                                           /* :145 */
            }
        }
    }
    if (hidden_out) memcpy(hidden_out, h, hidden * sizeof(float));
    /* compute_output_probs :162-188 */
    float* p = (float*)calloc(vocab, sizeof(float));
    for (size_t i = 0; i < vocab; ++i) {
        float acc = 0.0f;
        for (size_t j = 0; j < hidden; ++j) acc += h[j] * wout[i * hidden + j]; /* :166-173 */
        p[i] = acc;
    }
    float mx = p[0];
    for (size_t i = 1; i < vocab; ++i) if (p[i] > mx) mx = p[i]; /* max_element :176 */
    float sum = 0.0f;
    for (size_t i = 0; i < vocab; ++i) { p[i] = expf(p[i] - mx); sum += p[i]; } /* :178-181 */
    for (size_t i = 0; i < vocab; ++i) p[i] /= sum;                                /* :183-185 */
    /* top-k :72-92 (std::sort descending; tie order is unspecified in the
     * reference -- here ties go to the lower id) */
    for (size_t r = 0; r < k && r < vocab; ++r) {
        size_t best = (size_t)-1;
        for (size_t i = 0; i < vocab; ++i) {
            int taken = 0;
            for (size_t q = 0; q < r; ++q) if (ids[q] == i) { taken = 1; break; }
            if (taken) continue;
            if (best == (size_t)-1 || p[i] > p[best]) best = i;
        }
        ids[r] = (uint32_t)best;
        conf[r] = p[best];
    }
    free(hist); free(h); free(c); free(e); free(p);
}

/* compute_kv_address, speculative_prefetcher.cpp:153-160 */
uint64_t oracle_kv_address(uint32_t req_id, uint32_t layer_id, uint32_t position) {
    return ((uint64_t)req_id << 32) | ((uint64_t)layer_id << 16) | (uint64_t)position;
}

void oracle_depth_init(oracle_depth_t* d, unsigned depth) {
    memset(d, 0, sizeof(*d));
    d->depth = depth;
}

/* update_prediction_accuracy, speculative_prefetcher.cpp:99-120 */
unsigned oracle_depth_feedback(oracle_depth_t* d, int was_correct) {
    if (d->n == 100) {                      /* erase(begin()) once the window holds 100 */
        memmove(d->hist, d->hist + 1, 99 * sizeof(int));
        d->n = 99;
    }
    d->hist[d->n++] = was_correct ? 1 : 0;
    if (d->n >= 10) {
        double acc = 0.0;
        for (int i = d->n - 10; i < d->n; ++i) acc += d->hist[i];
        acc /= 10.0;
        if (acc > 0.95 && d->depth < 8) d->depth++;
        else if (acc < 0.85 && d->depth > 2) d->depth--;
    }
    return d->depth;
}

/* ---- tier residency policy (cxl_memory_manager.cpp:28-324) ------------------------------------ */
#define POL_NONE 0xffffffffffffffffull
struct oracle_policy {
    uint64_t n, cap[3], used[3];
    uint8_t* tier;            /* 0,1,2 or 255 */
    uint32_t* count;
    uint64_t *prev, *next;    /* LRU list links; POL_NONE = end */
    uint8_t* in_lru;
    uint64_t head, tail;      /* head = least recently used */
    oracle_policy_stats_t st;
};

oracle_policy_t* oracle_policy_new(uint64_t n_pages, uint64_t l1_cap, uint64_t l2_cap, uint64_t l3_cap) {
    oracle_policy_t* p = (oracle_policy_t*)calloc(1, sizeof(*p));
    if (!p) return NULL;
    p->n = n_pages;
    p->cap[0] = l1_cap; p->cap[1] = l2_cap; p->cap[2] = l3_cap;
    p->tier = (uint8_t*)malloc(n_pages ? n_pages : 1);
    p->count = (uint32_t*)calloc(n_pages ? n_pages : 1, sizeof(uint32_t));
    p->prev = (uint64_t*)malloc((n_pages ? n_pages : 1) * sizeof(uint64_t));
    p->next = (uint64_t*)malloc((n_pages ? n_pages : 1) * sizeof(uint64_t));
    p->in_lru = (uint8_t*)calloc(n_pages ? n_pages : 1, 1);
    memset(p->tier, 255, n_pages ? n_pages : 1);
    p->head = p->tail = POL_NONE;
    return p;
}

void oracle_policy_free(oracle_policy_t* p) {
    if (!p) return;
    free(p->tier); free(p->count); free(p->prev); free(p->next); free(p->in_lru); free(p);
}

static void pol_unlink(oracle_policy_t* p, uint64_t g) {
    if (!p->in_lru[g]) return;
    if (p->prev[g] != POL_NONE) p->next[p->prev[g]] = p->next[g]; else p->head = p->next[g];
    if (p->next[g] != POL_NONE) p->prev[p->next[g]] = p->prev[g]; else p->tail = p->prev[g];
    p->in_lru[g] = 0;
}

/* update_lru(): remove if present, append as most recently used  (:319-324) */
static void pol_to_back(oracle_policy_t* p, uint64_t g) {
    pol_unlink(p, g);
    p->prev[g] = p->tail; p->next[g] = POL_NONE;
    if (p->tail != POL_NONE) p->next[p->tail] = g; else p->head = g;
    p->tail = g;
    p->in_lru[g] = 1;
}

int oracle_policy_place(oracle_policy_t* p, uint64_t g, int tier) {
    if (g >= p->n || tier < 0 || tier > 2 || p->tier[g] != 255) return -1;
    /* only an L1 preference falls back, to L3  (:37-40) */
    if (tier == 0 && p->used[0] + 1 > p->cap[0]) tier = 2;
    p->tier[g] = (uint8_t)tier;
    p->used[tier]++;
    p->count[g] = 0;
    return tier;
}

void oracle_policy_release(oracle_policy_t* p, uint64_t g) {
    if (g >= p->n || p->tier[g] == 255) return;
    /* the reference drops the LRU entry only for an L1 page (:89-92); an L2/L3 page that was
     * touched keeps a dangling entry there.  Pages are indices here, so the entry is always dropped. */
    pol_unlink(p, g);
    p->used[p->tier[g]]--;
    p->tier[g] = 255;
    p->count[g] = 0;
}

void oracle_policy_touch(oracle_policy_t* p, uint64_t g) {
    if (g >= p->n || p->tier[g] == 255) return;
    p->count[g]++;
    if (p->tier[g] == 0) p->st.l1_hits++;
    else if (p->tier[g] == 1) p->st.l2_hits++;
    else p->st.l3_accesses++;
    pol_to_back(p, g);
}

int oracle_policy_is_hot(oracle_policy_t* p, uint64_t g) {
    if (g >= p->n || p->tier[g] == 255) return 0;
    return p->count[g] > 10;
}

int oracle_policy_demote(oracle_policy_t* p, uint64_t g) {
    if (g >= p->n || p->tier[g] == 255 || p->tier[g] == 2) return 0;
    if (p->tier[g] == 0) {
        pol_unlink(p, g);
        p->st.migrations_l1_to_l3++;
    }
    p->used[p->tier[g]]--;
    p->tier[g] = 2;
    p->used[2]++;
    return 1;
}

int oracle_policy_promote(oracle_policy_t* p, uint64_t g, uint64_t* evicted) {
    if (evicted) *evicted = POL_NONE;
    if (g >= p->n || p->tier[g] == 255 || p->tier[g] == 0) return 0;
    if (p->used[0] + 1 > p->cap[0]) {
        /* evict_l1_lru (:285-293), repeated until an L1 page has been demoted */
        while (p->head != POL_NONE) {
            const uint64_t v = p->head;
            pol_unlink(p, v);
            if (p->tier[v] == 0) {
                oracle_policy_demote(p, v);
                if (evicted) *evicted = v;
                break;
            }
        }
    }
    if (p->tier[g] == 2) p->st.migrations_l3_to_l1++;
    p->used[p->tier[g]]--;
    p->tier[g] = 0;
    p->used[0]++;
    pol_to_back(p, g);
    return 1;
}

int oracle_policy_tier(const oracle_policy_t* p, uint64_t g) { return g < p->n ? p->tier[g] : 255; }

size_t oracle_policy_lru(const oracle_policy_t* p, uint64_t* out, size_t cap) {
    size_t k = 0;
    for (uint64_t g = p->head; g != POL_NONE; g = p->next[g]) {
        if (k < cap) out[k] = g;
        ++k;
    }
    return k;
}

/* batch forms: the single-page calls above, in order */
void oracle_policy_touch_n(oracle_policy_t* p, const uint64_t* pages, size_t n) {
    for (size_t i = 0; i < n; ++i) oracle_policy_touch(p, pages[i]);
}

void oracle_policy_place_n(oracle_policy_t* p, const uint64_t* pages, size_t n, int tier, int32_t* out) {
    for (size_t i = 0; i < n; ++i) {
        const int t = oracle_policy_place(p, pages[i], tier);
        if (out) out[i] = t;
    }
}

void oracle_policy_release_n(oracle_policy_t* p, const uint64_t* pages, size_t n) {
    for (size_t i = 0; i < n; ++i) oracle_policy_release(p, pages[i]);
}

void oracle_policy_demote_n(oracle_policy_t* p, const uint64_t* pages, size_t n, uint8_t* ok) {
    for (size_t i = 0; i < n; ++i) {
        const int r = oracle_policy_demote(p, pages[i]);
        if (ok) ok[i] = (uint8_t)r;
    }
}

void oracle_policy_is_hot_n(oracle_policy_t* p, const uint64_t* pages, size_t n, uint8_t* hot) {
    for (size_t i = 0; i < n; ++i) hot[i] = (uint8_t)oracle_policy_is_hot(p, pages[i]);
}

size_t oracle_policy_promote_n(oracle_policy_t* p, const uint64_t* pages, size_t n, uint8_t* ok, uint64_t* evicted) {
    size_t k = 0;
    for (size_t i = 0; i < n; ++i) {
        uint64_t ev;
        const int r = oracle_policy_promote(p, pages[i], &ev);
        if (ok) ok[i] = (uint8_t)r;
        if (ev != POL_NONE) {
            if (evicted) evicted[k] = ev;
            ++k;
        }
    }
    return k;
}

void oracle_policy_tiers(const oracle_policy_t* p, uint8_t* out) {
    for (uint64_t g = 0; g < p->n; ++g) out[g] = p->tier[g];
}

void oracle_policy_stats(const oracle_policy_t* p, oracle_policy_stats_t* out) {
    *out = p->st;
    const uint64_t t1 = out->l1_hits + out->l1_misses, t2 = out->l2_hits + out->l2_misses;
    out->l1_hit_rate = t1 ? (double)out->l1_hits / (double)t1 : 0.0;
    out->l2_hit_rate = t2 ? (double)out->l2_hits / (double)t2 : 0.0;
    out->l1_pages = p->used[0]; out->l2_pages = p->used[1]; out->l3_pages = p->used[2];
}

uint64_t oracle_fnv1a64(const void* p, size_t n) {
    const uint8_t* b = (const uint8_t*)p;
    uint64_t h = 0xcbf29ce484222325ULL;
    for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 0x100000001b3ULL; }
    return h;
}


/* ------------------------------------------------------------------------ */
/* CXLMemoryManager address map: src/cxl_memory/cxl_memory_manager.cpp:8-128  */
/* ------------------------------------------------------------------------ */
struct oracle_mm {
    uint64_t cap[3], page, next_va, next_pa[3], n_alloc[3];
    uint64_t n_pages, cap_pages;   /* page entries, indexed by (va - 0x100000000) / page */
    uint64_t* pa;                  /* 0 = no entry */
    uint8_t* tier;
    uint8_t* base;                 /* 1 = first page of an allocation (the address the tier lists hold) */
};

oracle_mm_t* oracle_mm_new(uint64_t l1_bytes, uint64_t l2_bytes, uint64_t l3_bytes, uint64_t page_size) {
    oracle_mm_t* m = (oracle_mm_t*)calloc(1, sizeof(*m));
    if (!m) return NULL;
    m->cap[0] = l1_bytes; m->cap[1] = l2_bytes; m->cap[2] = l3_bytes;
    m->page = page_size;
    m->next_va = 0x100000000ULL;                                        /* :18 */
    m->next_pa[0] = 0x8000000000ULL; m->next_pa[1] = 0x10000000000ULL; m->next_pa[2] = 0x20000000000ULL;   /* :19-21 */
    return m;
}

void oracle_mm_free(oracle_mm_t* m) {
    if (!m) return;
    free(m->pa); free(m->tier); free(m->base); free(m);
}

uint64_t oracle_mm_allocate(oracle_mm_t* m, uint64_t size_bytes, uint32_t layer, int tier) {
    (void)layer;
    const uint64_t pages = (size_bytes + m->page - 1) / m->page, bytes = pages * m->page;      /* :32-33 */
    if (tier == 0 && m->n_alloc[0] * m->page + bytes > m->cap[0]) tier = 2;                     /* :37-39, :295-316 */
    const uint64_t va = m->next_va, pa = m->next_pa[tier];
    m->next_pa[tier] += bytes;
    m->n_alloc[tier] += 1;                                                                      /* lX_pages_.push_back(va) */
    const uint64_t first = (va - 0x100000000ULL) / m->page;
    if (first + pages > m->cap_pages) {
        uint64_t nc = m->cap_pages ? m->cap_pages * 2 : 1024;
        while (nc < first + pages) nc *= 2;
        m->pa = (uint64_t*)realloc(m->pa, nc * sizeof(uint64_t));
        m->tier = (uint8_t*)realloc(m->tier, nc);
        m->base = (uint8_t*)realloc(m->base, nc);
        memset(m->pa + m->cap_pages, 0, (nc - m->cap_pages) * sizeof(uint64_t));
        memset(m->tier + m->cap_pages, 255, nc - m->cap_pages);
        memset(m->base + m->cap_pages, 0, nc - m->cap_pages);
        m->cap_pages = nc;
    }
    for (uint64_t i = 0; i < pages; ++i) {                                                      /* :62-75 */
        m->pa[first + i] = pa + i * m->page;
        m->tier[first + i] = (uint8_t)tier;
        m->base[first + i] = (i == 0);
    }
    if (first + pages > m->n_pages) m->n_pages = first + pages;
    m->next_va += bytes;                                                                        /* :77 */
    return va;
}

void oracle_mm_deallocate(oracle_mm_t* m, uint64_t va) {                                        /* :81-104 */
    if (va < 0x100000000ULL || (va - 0x100000000ULL) % m->page) return;                          /* the map is keyed by page addresses */
    const uint64_t i = (va - 0x100000000ULL) / m->page;
    if (i >= m->n_pages || m->pa[i] == 0) return;
    if (m->base[i] && m->n_alloc[m->tier[i]]) m->n_alloc[m->tier[i]] -= 1;   /* std::remove of va from the tier list: it holds base addresses only */
    m->pa[i] = 0;
    m->tier[i] = 255;
    m->base[i] = 0;
}

uint64_t oracle_mm_translate(const oracle_mm_t* m, uint64_t va) {                               /* :106-117 */
    const uint64_t page_addr = (va / m->page) * m->page;
    if (page_addr < 0x100000000ULL) return 0;
    const uint64_t i = (page_addr - 0x100000000ULL) / m->page;
    if (i >= m->n_pages || m->pa[i] == 0) return 0;
    return m->pa[i] + (va - page_addr);
}

int oracle_mm_is_in_cache(const oracle_mm_t* m, uint64_t va, int tier) {                        /* :119-128 */
    const uint64_t page_addr = (va / m->page) * m->page;
    if (page_addr < 0x100000000ULL) return 0;
    const uint64_t i = (page_addr - 0x100000000ULL) / m->page;
    if (i >= m->n_pages || m->pa[i] == 0) return 0;
    return m->tier[i] == tier;
}
